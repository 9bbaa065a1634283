// smc_soa.cpp -- host-side batch packer (include/smc_soa.h): gathers the reads of a batch out of the decoded BAM and writes
// them in the compact wire encodings of smc_reads_soa, one threaded pass, into caller-owned (pinned) buffers.
#include "../../include/smc_soa.h"

#include <algorithm>
#include <cstring>
#include <memory>
#include <new>
#include <vector>

#include "smc_host.h"

using smc_host::n_threads;

namespace {

template <class F> void par_for(size_t n, int threads, F&& f) {    // f(begin, end, thread); inline below 4096 items
    smc_host::for_ranges(n, n < 4096 ? 1 : threads, f);
}

struct Exc { uint32_t read, pos; uint8_t nib; };

// SMC_SOA_TIMING=1: phase times on stderr
smc_host::PhaseTimer phase_timer() { return smc_host::PhaseTimer("SMC_SOA_TIMING", "smc_soa"); }

}  // namespace

struct smc_soa_pack {
    smc_soa_view v;
    const int64_t* idx;
    int64_t n;
    smc_soa_pack_opts o;
    int threads;
    std::unique_ptr<int64_t[]> seq_off, qual_off, cig_off; // n + 1 each: offsets inside the packed arrays (not zero-filled)
    uint32_t frag_lo = 0;
    std::vector<uint32_t> frag_rank;                       // rank of parent id frag_lo + i among the ids of the batch
    std::vector<uint16_t> qpair;                           // quality pair (q0 | q1 << 8) -> its two codes (c0 | c1 << qual_bits), bit 15: no code
    uint8_t seq_code[256], seq_odd[256];                   // source byte (two bases) -> two 2-bit codes; ... holds a non-ACGT base
    std::vector<uint32_t> exc_read, exc_pos;
    std::vector<uint8_t> exc_nib;
    int64_t src(int64_t k) const { return idx ? idx[k] : k; }
    int32_t len(int64_t r) const { const int32_t l = v.store_len ? v.store_len[r] : v.l_seq[r]; return l > 0 ? l : 0; }
};

extern "C" int smc_soa_qual_hist(const smc_soa_view* v, int threads, uint64_t hist[256]) {
    if (!v || !hist || v->n_reads < 0) return SMC_SOA_E_ARG;
    const int T = n_threads(threads);
    std::vector<std::vector<uint64_t>> part((size_t)T, std::vector<uint64_t>(256, 0));
    par_for((size_t)v->n_reads, T, [&](size_t a, size_t e, int t) {
        // four private tables: binned qualities hit the same few counters, one table would serialise on store forwarding
        uint32_t h[4][256];
        memset(h, 0, sizeof(h));
        uint64_t* out = part[(size_t)t].data();
        uint64_t since = 0;
        for (size_t r = a; r < e; ++r) {
            const int32_t l = v->store_len ? v->store_len[r] : v->l_seq[r];
            const uint8_t* q = v->qual + v->qual_off[r];
            int32_t i = 0;
            for (; i + 4 <= l; i += 4) { ++h[0][q[i]]; ++h[1][q[i + 1]]; ++h[2][q[i + 2]]; ++h[3][q[i + 3]]; }
            for (; i < l; ++i) ++h[0][q[i]];
            since += (uint64_t)(l > 0 ? l : 0);
            if (since > (1u << 30)) {                                  // flush before a 32-bit counter can wrap
                for (int c = 0; c < 256; ++c) { out[c] += (uint64_t)h[0][c] + h[1][c] + h[2][c] + h[3][c]; }
                memset(h, 0, sizeof(h)); since = 0;
            }
        }
        for (int c = 0; c < 256; ++c) out[c] += (uint64_t)h[0][c] + h[1][c] + h[2][c] + h[3][c];
    });
    for (int c = 0; c < 256; ++c) { hist[c] = 0; for (int t = 0; t < T; ++t) hist[c] += part[(size_t)t][(size_t)c]; }
    return SMC_SOA_OK;
}

extern "C" int smc_soa_ref_end(const smc_soa_view* v, int threads, int64_t* ref_end) {
    if (!v || v->n_reads < 0 || (v->n_reads > 0 && !ref_end)) return SMC_SOA_E_ARG;
    par_for((size_t)v->n_reads, n_threads(threads), [&](size_t a, size_t e, int) {
        for (size_t r = a; r < e; ++r) {
            const uint32_t* c = v->cigar + v->cigar_off[r];
            int64_t span = 0;
            for (int k = 0, nc = v->n_cigar[r]; k < nc; ++k) {
                const uint32_t op = c[k] & 15u;
                if (op == 0u || op == 2u || op == 3u || op == 7u || op == 8u) span += (int64_t)(c[k] >> 4);
            }
            ref_end[r] = (int64_t)v->pos[r] + span;
        }
    });
    return SMC_SOA_OK;
}

extern "C" int smc_soa_order_stats(const smc_soa_view* v, int threads, int64_t* ref_end, int64_t stats[2]) {
    if (!v || !stats || v->n_reads < 0 || (v->n_reads > 0 && !ref_end)) return SMC_SOA_E_ARG;
    const int T = n_threads(threads);
    std::vector<int64_t> span((size_t)T, 0);
    std::vector<int> unsorted((size_t)T, 0);
    par_for((size_t)v->n_reads, T, [&](size_t a, size_t e, int t) {
        int64_t longest = 0;
        int bad = 0;
        for (size_t r = a; r < e; ++r) {
            const uint32_t* c = v->cigar + v->cigar_off[r];
            int64_t sp = 0;
            for (int k = 0, nc = v->n_cigar[r]; k < nc; ++k) {
                const uint32_t op = c[k] & 15u;
                if (op == 0u || op == 2u || op == 3u || op == 7u || op == 8u) sp += (int64_t)(c[k] >> 4);
            }
            ref_end[r] = (int64_t)v->pos[r] + sp;
            if (sp > longest) longest = sp;
            if (r > 0 && (v->ref_id[r] < v->ref_id[r - 1] || (v->ref_id[r] == v->ref_id[r - 1] && v->pos[r] < v->pos[r - 1]))) bad = 1;
        }
        span[(size_t)t] = longest; unsorted[(size_t)t] = bad;
    });
    stats[0] = 1; stats[1] = 0;
    for (int t = 0; t < T; ++t) { if (unsorted[(size_t)t]) stats[0] = 0; if (span[(size_t)t] > stats[1]) stats[1] = span[(size_t)t]; }
    return SMC_SOA_OK;
}

extern "C" int smc_soa_pack_begin(const smc_soa_view* v, const int64_t* idx, int64_t n_idx, const smc_soa_pack_opts* opts,
                                  smc_soa_pack** out, smc_soa_pack_sizes* sizes) {
    if (!v || !opts || !out || !sizes || v->n_reads < 0 || (idx && n_idx < 0)) return SMC_SOA_E_ARG;
    if ((opts->scalar_bits != 8 && opts->scalar_bits != 16 && opts->scalar_bits != 32) || (opts->qual_bits != 2 && opts->qual_bits != 4 && opts->qual_bits != 8) ||
        (opts->seq_bits != 2 && opts->seq_bits != 4) || (opts->ref_id_bits != 8 && opts->ref_id_bits != 32) ||
        (opts->umi_bits != 32 && opts->umi_bits != 64) || ((v->store_lo == nullptr) != (v->store_len == nullptr)))
        return SMC_SOA_E_ARG;
    smc_soa_pack* h = new (std::nothrow) smc_soa_pack();
    if (!h) return SMC_SOA_E_MEM;
    h->v = *v; h->idx = idx; h->n = idx ? n_idx : v->n_reads; h->o = *opts; h->threads = n_threads(opts->threads);
    const int64_t n = h->n;
    auto pt = phase_timer();
    try {
        h->seq_off.reset(new int64_t[(size_t)n + 1]); h->qual_off.reset(new int64_t[(size_t)n + 1]); h->cig_off.reset(new int64_t[(size_t)n + 1]);
        h->seq_off[0] = h->qual_off[0] = h->cig_off[0] = 0;      // the sizes pass writes every other entry
    } catch (...) { delete h; return SMC_SOA_E_MEM; }
    const int T = h->threads;
    const int qb = opts->qual_bits, sb = opts->seq_bits;
    pt.lap("begin: alloc offsets");
    // pass 1: per-read sizes into slot k + 1, range checks, the span of fragment ids
    std::vector<int> bad((size_t)T, 0);
    std::vector<uint32_t> fmin((size_t)T, 0xffffffffu), fmax((size_t)T, 0u);
    par_for((size_t)n, T, [&](size_t a, size_t e, int t) {
        int64_t prev = a ? h->src((int64_t)a - 1) : -1;
        uint32_t lo = 0xffffffffu, hi = 0u;                          // thread-local: the per-thread slots share cache lines
        for (size_t k = a; k < e; ++k) {
            const int64_t r = h->src((int64_t)k);
            if (r <= prev || r >= v->n_reads) { bad[(size_t)t] = 1; return; }
            prev = r;
            const int64_t l = h->len(r);
            h->seq_off[k + 1] = sb == 2 ? (l + 3) / 4 : (l + 1) / 2;
            h->qual_off[k + 1] = qb == 8 ? l : (l * qb + 7) / 8;
            h->cig_off[k + 1] = v->n_cigar[r];
            if (opts->scalar_bits != 32) {
                const uint32_t lim = opts->scalar_bits == 16 ? 65536u : 256u;
                const bool ok = (uint32_t)v->nm[r] < lim && (uint32_t)v->l_seq[r] < lim &&
                                (!v->store_lo || ((uint32_t)v->store_lo[r] < lim && (uint32_t)v->store_len[r] < lim));
                if (!ok) { bad[(size_t)t] = 1; return; }
            }
            if ((opts->ref_id_bits == 8 && (uint32_t)v->ref_id[r] >= 256u) || (opts->umi_bits == 32 && (v->umi[r] >> 32) != 0)) { bad[(size_t)t] = 1; return; }
            lo = std::min(lo, v->frag_id[r]); hi = std::max(hi, v->frag_id[r]);
        }
        fmin[(size_t)t] = lo; fmax[(size_t)t] = hi;
    });
    for (int t = 0; t < T; ++t) if (bad[(size_t)t]) { delete h; return SMC_SOA_E_RANGE; }
    pt.lap("begin: sizes pass");
    // prefix sums: every range scans its own slice, the range totals are scanned serially, every range adds its base
    {
        struct Tot { int64_t s, q, c; };
        std::vector<Tot> tot((size_t)T + 1, Tot{0, 0, 0});
        const int tasks = (size_t)n < 65536 ? 1 : T;
        smc_host::for_ranges((size_t)n, tasks, [&](size_t a, size_t e, int t) {
            Tot run{0, 0, 0};
            for (size_t k = a; k < e; ++k) {
                run.s += h->seq_off[k + 1]; run.q += h->qual_off[k + 1]; run.c += h->cig_off[k + 1];
                h->seq_off[k + 1] = run.s; h->qual_off[k + 1] = run.q; h->cig_off[k + 1] = run.c;
            }
            tot[(size_t)t + 1] = run;
        });
        for (int t = 0; t < tasks; ++t) { tot[(size_t)t + 1].s += tot[(size_t)t].s; tot[(size_t)t + 1].q += tot[(size_t)t].q; tot[(size_t)t + 1].c += tot[(size_t)t].c; }
        if (tasks > 1)
            smc_host::for_ranges((size_t)n, tasks, [&](size_t a, size_t e, int t) {
                if (t == 0) return;
                const Tot b = tot[(size_t)t];
                for (size_t k = a; k < e; ++k) { h->seq_off[k + 1] += b.s; h->qual_off[k + 1] += b.q; h->cig_off[k + 1] += b.c; }
            });
    }
    pt.lap("begin: prefix sums");
    // dense fragment ids in the old relative order: mark the ids of the batch, count them in order
    if (n > 0) {
        uint32_t lo = 0xffffffffu, hi = 0;
        for (int t = 0; t < T; ++t) { lo = std::min(lo, fmin[(size_t)t]); hi = std::max(hi, fmax[(size_t)t]); }
        h->frag_lo = lo;
        try { h->frag_rank.assign((size_t)(hi - lo) + 1, 0u); } catch (...) { delete h; return SMC_SOA_E_MEM; }
        par_for((size_t)n, T, [&](size_t a, size_t e, int) {
            for (size_t k = a; k < e; ++k) h->frag_rank[v->frag_id[h->src((int64_t)k)] - lo] = 1u;      // racing writers store the same value
        });
        uint32_t run = 0;
        for (auto& f : h->frag_rank) { const uint32_t m = f; f = run; run += m; }
    }
    pt.lap("begin: fragment ranks");
    {   // look-up tables of the fill pass
        uint8_t code2[16] = {0}, plain[16] = {0};
        code2[2] = 1; code2[4] = 2; code2[8] = 3; plain[1] = plain[2] = plain[4] = plain[8] = 1;
        for (int b = 0; b < 256; ++b) {
            h->seq_code[b] = (uint8_t)(code2[b >> 4] | (code2[b & 15] << 2));
            h->seq_odd[b] = (uint8_t)(!plain[b >> 4] || !plain[b & 15]);
        }
        if (qb != 8) {
            try { h->qpair.assign(65536, 0); } catch (...) { delete h; return SMC_SOA_E_MEM; }
            for (int q1 = 0; q1 < 256; ++q1)
                for (int q0 = 0; q0 < 256; ++q0) {
                    const uint8_t c0 = opts->code_of[q0], c1 = opts->code_of[q1];
                    h->qpair[(size_t)(q0 | (q1 << 8))] = (c0 == 0xffu || c1 == 0xffu) ? (uint16_t)0x8000u : (uint16_t)(c0 | (c1 << qb));
                }
        }
    }
    pt.lap("begin: tables");
    sizes->n_reads = n; sizes->seq_bytes = h->seq_off[(size_t)n]; sizes->qual_bytes = h->qual_off[(size_t)n]; sizes->n_cigar_words = h->cig_off[(size_t)n];
    *out = h;
    return SMC_SOA_OK;
}

extern "C" int smc_soa_pack_fill(smc_soa_pack* h, const smc_soa_pack_bufs* B, smc_soa_pack_exc* exc) {
    if (!h || !B) return SMC_SOA_E_ARG;
    const smc_soa_view& v = h->v;
    const int64_t n = h->n;
    const bool has_store = v.store_lo != nullptr;
    if (n > 0 && (!B->ref_id || !B->pos || !B->flag || !B->mapq || !B->nm || !B->l_seq || !B->n_cigar || !B->umi || !B->frag_id ||
                  (has_store && (!B->store_lo || !B->store_len)) || (h->seq_off[(size_t)n] && !B->seq) || (h->qual_off[(size_t)n] && !B->qual) ||
                  (h->cig_off[(size_t)n] && !B->cigar)))
        return SMC_SOA_E_ARG;
    const int T = h->threads, qb = h->o.qual_bits, sb = h->o.seq_bits;
    const bool s16 = h->o.scalar_bits == 16, s8 = h->o.scalar_bits == 8, ref8 = h->o.ref_id_bits == 8, umi32 = h->o.umi_bits == 32;
    // BAM nibble -> 2-bit code (A 1, C 2, G 4, T 8); everything else travels as code 0 plus an exception
    uint8_t code2[16], plain[16];
    for (int i = 0; i < 16; ++i) { code2[i] = 0; plain[i] = 0; }
    code2[1] = 0; code2[2] = 1; code2[4] = 2; code2[8] = 3; plain[1] = plain[2] = plain[4] = plain[8] = 1;
    std::vector<std::vector<Exc>> excs((size_t)T);
    std::vector<int> bad((size_t)T, 0);
    auto pt = phase_timer();
    par_for((size_t)n, T, [&](size_t a, size_t e, int t) {
        std::vector<Exc>& ex = excs[(size_t)t];
        for (size_t k = a; k < e; ++k) {
            const int64_t r = h->src((int64_t)k);
            if (ref8) ((uint8_t*)B->ref_id)[k] = (uint8_t)v.ref_id[r]; else ((int32_t*)B->ref_id)[k] = v.ref_id[r];
            if (umi32) ((uint32_t*)B->umi)[k] = (uint32_t)v.umi[r]; else ((uint64_t*)B->umi)[k] = v.umi[r];
            B->pos[k] = v.pos[r]; B->flag[k] = v.flag[r]; B->mapq[k] = v.mapq[r];
            B->n_cigar[k] = v.n_cigar[r];
            B->frag_id[k] = h->frag_rank[v.frag_id[r] - h->frag_lo];
            if (s8) {
                ((uint8_t*)B->nm)[k] = (uint8_t)v.nm[r]; ((uint8_t*)B->l_seq)[k] = (uint8_t)v.l_seq[r];
                if (has_store) { ((uint8_t*)B->store_lo)[k] = (uint8_t)v.store_lo[r]; ((uint8_t*)B->store_len)[k] = (uint8_t)v.store_len[r]; }
            } else if (s16) {
                ((uint16_t*)B->nm)[k] = (uint16_t)v.nm[r]; ((uint16_t*)B->l_seq)[k] = (uint16_t)v.l_seq[r];
                if (has_store) { ((uint16_t*)B->store_lo)[k] = (uint16_t)v.store_lo[r]; ((uint16_t*)B->store_len)[k] = (uint16_t)v.store_len[r]; }
            } else {
                ((int32_t*)B->nm)[k] = v.nm[r]; ((int32_t*)B->l_seq)[k] = v.l_seq[r];
                if (has_store) { ((int32_t*)B->store_lo)[k] = v.store_lo[r]; ((int32_t*)B->store_len)[k] = v.store_len[r]; }
            }
            if (B->seq_poff) B->seq_poff[k] = h->seq_off[k];
            const int32_t nc = v.n_cigar[r];
            if (nc) std::memcpy(B->cigar + h->cig_off[k], v.cigar + v.cigar_off[r], (size_t)nc * 4);
            const int32_t l = h->len(r);
            const uint8_t* s = v.seq + v.seq_off[r];
            uint8_t* so = B->seq + h->seq_off[k];
            if (sb == 4) {
                if (l) std::memcpy(so, s, (size_t)(l + 1) / 2);
            } else {
                const int32_t full = l & ~3;                         // four bases = two source bytes -> one output byte
                for (int32_t i = 0; i < full; i += 4) {
                    const uint32_t b0 = s[i >> 1], b1 = s[(i >> 1) + 1];
                    so[i >> 2] = (uint8_t)(h->seq_code[b0] | (h->seq_code[b1] << 4));
                    if (h->seq_odd[b0] | h->seq_odd[b1]) {
                        const uint32_t nib[4] = {b0 >> 4, b0 & 15u, b1 >> 4, b1 & 15u};
                        for (int j = 0; j < 4; ++j) if (!plain[nib[j]]) ex.push_back(Exc{(uint32_t)k, (uint32_t)(i + j), (uint8_t)nib[j]});
                    }
                }
                if (full < l) {                                      // the last 1-3 bases; past the end: 'A' (code 0)
                    const int32_t i = full;
                    const uint32_t b0 = s[i >> 1], b1 = i + 2 < l ? s[(i >> 1) + 1] : 0x11u;
                    uint32_t nib[4] = {b0 >> 4, b0 & 15u, b1 >> 4, b1 & 15u};
                    if (i + 1 >= l) nib[1] = 1u;
                    if (i + 3 >= l) nib[3] = 1u;
                    uint32_t o = 0;
                    for (int j = 0; j < 4; ++j) {
                        o |= (uint32_t)code2[nib[j]] << (2 * j);
                        if (!plain[nib[j]]) ex.push_back(Exc{(uint32_t)k, (uint32_t)(i + j), (uint8_t)nib[j]});
                    }
                    so[i >> 2] = (uint8_t)o;
                }
            }
            const uint8_t* q = v.qual + v.qual_off[r];
            uint8_t* qo = B->qual + h->qual_off[k];
            if (qb == 8) {
                if (l) std::memcpy(qo, q, (size_t)l);
            } else {
                const int per = 8 / qb;
                const uint8_t* code_of = h->o.code_of;
                const uint16_t* qp = h->qpair.data();
                const int32_t full = l - l % per;
                uint32_t invalid = 0;
                if (qb == 2) {
                    for (int32_t i = 0; i < full; i += 4) {
                        const uint32_t a = qp[q[i] | (q[i + 1] << 8)], b = qp[q[i + 2] | (q[i + 3] << 8)];
                        invalid |= a | b;
                        qo[i >> 2] = (uint8_t)(a | (b << 4));
                    }
                } else {
                    for (int32_t i = 0; i < full; i += 2) {
                        const uint32_t a = qp[q[i] | (q[i + 1] << 8)];
                        invalid |= a;
                        qo[i >> 1] = (uint8_t)a;
                    }
                }
                if (full < l) {
                    uint32_t o = 0;
                    for (int j = 0; full + j < l; ++j) {
                        const uint32_t c = code_of[q[full + j]];
                        if (c == 0xffu) invalid |= 0x8000u;
                        o |= (c & 15u) << (qb * j);
                    }
                    qo[full / per] = (uint8_t)o;
                }
                if (invalid & 0x8000u) { bad[(size_t)t] = 1; return; }
            }
        }
    });
    for (int t = 0; t < T; ++t) if (bad[(size_t)t]) return SMC_SOA_E_RANGE;
    pt.lap("fill: pass");
    if (B->seq_poff) B->seq_poff[n] = h->seq_off[(size_t)n];
    size_t ne = 0;
    for (auto& ex : excs) ne += ex.size();
    try { h->exc_read.resize(ne); h->exc_pos.resize(ne); h->exc_nib.resize(ne); } catch (...) { return SMC_SOA_E_MEM; }
    size_t o = 0;
    for (auto& ex : excs) for (const Exc& x : ex) { h->exc_read[o] = x.read; h->exc_pos[o] = x.pos; h->exc_nib[o] = x.nib; ++o; }   // thread order = read order
    pt.lap("fill: exceptions");
    if (exc) { exc->n = (int64_t)ne; exc->read = h->exc_read.data(); exc->pos = h->exc_pos.data(); exc->nib = h->exc_nib.data(); }
    return SMC_SOA_OK;
}

extern "C" void smc_soa_pack_end(smc_soa_pack* h) { delete h; }
