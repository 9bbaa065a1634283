// Host-side output stage (include/smc_rows.h): device results -> the reference's text rows, repeat filters, called-variant
// lines.  Restates smCounter.py:552-600 (row), :751-785 (repeat filters), :832-891 (writers) over the smc_out arrays; the
// Python-2 number formatting (round() half away from zero on the exact binary value, str(float) = shortest form of the rounded
// value) is done in exact integer arithmetic.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/smc_b200.h"
#include "../../include/smc_rows.h"
#include "smc_host.h"

namespace {

// bits of smc_out::fl1 / fl2 that the row needs (include/smc_b200.h)
constexpr uint32_t F_LM = SMC_F_LM, F_LSM = SMC_F_LSM, F_DP = SMC_F_DP, F_SB = SMC_F_SB, F_LOWQ = SMC_F_LOWQ, F_R1CP = SMC_F_R1CP,
                   F_R2CP = SMC_F_R2CP, F_PRIMERCP = SMC_F_PRIMERCP, F_HPGATE = SMC_F_HPGATE, F_EVALUATED = SMC_F_EVALUATED;

// round(x * scale) with ties away from zero, decided on the exact binary value of x (Python-2 round(x, nd), scale = 10^nd).
// x >= 0 and finite.
uint64_t round_scaled(double x, uint32_t scale) {
    if (!(x > 0.0)) return 0;
    int e;
    const double m = std::frexp(x, &e);                       // x = m * 2^e, 0.5 <= m < 1
    const uint64_t M = (uint64_t)std::ldexp(m, 53);           // exact 53-bit integer
    const int E = e - 53;                                     // x = M * 2^E
    const unsigned __int128 P = (unsigned __int128)M * scale;
    if (E >= 0) return E < 40 ? (uint64_t)(P << E) : ~0ull;
    const int s = -E;
    if (s >= 120) return 0;
    unsigned __int128 q = P >> s;
    const unsigned __int128 rem = P & (((unsigned __int128)1 << s) - 1), half = (unsigned __int128)1 << (s - 1);
    if (rem >= half) ++q;
    return (uint64_t)q;
}

inline void put_uint(std::string& o, uint64_t v) {
    char b[24]; int n = 0;
    do { b[n++] = (char)('0' + v % 10); v /= 10; } while (v);
    while (n) o.push_back(b[--n]);
}
inline void put_int(std::string& o, int64_t v) {
    if (v < 0) { o.push_back('-'); put_uint(o, (uint64_t)(-v)); } else put_uint(o, (uint64_t)v);
}
// Python-2 str() of the double nearest to k / 10^nd (nd = 2 or 4): shortest decimal, at least one fractional digit
void put_scaled(std::string& o, uint64_t k, int nd) {
    const uint64_t scale = nd == 2 ? 100ull : 10000ull;
    if (k >= 100000000000ull * scale / 100ull && nd == 2) {               // >= 1e9: '%.12g' territory, leave it to printf
        char b[64];
        std::snprintf(b, sizeof b, "%.12g", (double)k / 100.0);
        o += b;
        if (!std::strpbrk(b, ".en")) o += ".0";
        return;
    }
    put_uint(o, k / scale);
    o.push_back('.');
    uint64_t f = k % scale;
    char d[4];
    for (int i = nd - 1; i >= 0; --i) { d[i] = (char)('0' + f % 10); f /= 10; }
    int n = nd;
    while (n > 1 && d[n - 1] == '0') --n;
    o.append(d, (size_t)n);
}
inline uint64_t frac4(int64_t num, int64_t den) { return (num <= 0 || den <= 0) ? 0 : round_scaled((double)num / (double)den, 10000); }

struct Regions {              // per contig: [first, last) into the flat arrays, and the running maximum of the upper ends
    std::vector<int64_t> first, last;
    std::vector<int64_t> pmax;
    const int64_t *lo = nullptr, *hi = nullptr;
    void build(int32_t n_chroms, int64_t n, const int32_t* chrom, const int64_t* lo_, const int64_t* hi_) {
        lo = lo_; hi = hi_;
        first.assign((size_t)n_chroms, 0); last.assign((size_t)n_chroms, 0);
        pmax.resize((size_t)n);
        for (int64_t r = 0; r < n;) {
            const int32_t c = chrom[r];
            int64_t e = r;
            int64_t mx = INT64_MIN;
            while (e < n && chrom[e] == c) { mx = std::max(mx, hi_[e]); pmax[(size_t)e] = mx; ++e; }
            if (c >= 0 && c < n_chroms && last[(size_t)c] == 0) { first[(size_t)c] = r; last[(size_t)c] = e; }
            r = e;
        }
    }
    // first region in list order with lo < pos <= hi (smCounter.py:773-776, :779-782); regions of a contig are sorted by lo
    int64_t first_hit(int32_t c, int64_t pos) const {
        if (c < 0 || (size_t)c >= first.size()) return -1;
        const int64_t a = first[(size_t)c], b = last[(size_t)c];
        if (a >= b) return -1;
        const int64_t k = std::lower_bound(lo + a, lo + b, pos) - lo;                  // regions [a, k) have lo < pos
        const int64_t i = std::lower_bound(pmax.begin() + a, pmax.begin() + k, pos) - pmax.begin();   // first with max(hi) >= pos
        return i < k ? i : -1;
    }
};

struct Ctx {
    const smc_rows_in* in;
    Regions trf, rm;
};

struct Chunk {
    std::string all, cut, vcf;
    std::vector<int64_t> all_len, cut_len, vcf_len;
    int status = SMC_ROWS_OK; int64_t bad_row = -1; uint32_t bad_status = 0;
};

struct Allele { const char* ref; size_t ref_n; const char* alt; size_t alt_n; const char* vtype; bool is_del_word; };

// convertToVcf (smCounter.py:103-117) on the allele string `name`
Allele convert_to_vcf(const char* origRef, const char* name, size_t n) {
    Allele a{origRef, 1, name, n, ".", false};
    if (n == 1) { a.vtype = "SNP"; return a; }
    if (n == 3 && std::memcmp(name, "DEL", 3) == 0) { a.vtype = "SDEL"; a.is_del_word = true; return a; }
    const char* p1 = (const char*)std::memchr(name, '|', n);
    if (p1 && ((p1 - name == 3 && (std::memcmp(name, "DEL", 3) == 0 || std::memcmp(name, "INS", 3) == 0)))) {
        const char* p2 = (const char*)std::memchr(p1 + 1, '|', n - (size_t)(p1 + 1 - name));
        if (p2) { a.vtype = "INDEL"; a.ref = p1 + 1; a.ref_n = (size_t)(p2 - p1 - 1); a.alt = p2 + 1; a.alt_n = n - (size_t)(p2 + 1 - name); }
    }
    return a;
}
const char* lower_type(const char* t) {
    if (!std::strcmp(t, "SNP")) return "snp";
    if (!std::strcmp(t, "SDEL")) return "sdel";
    if (!std::strcmp(t, "INDEL")) return "indel";
    return t;
}

// FILTER accumulator of filterVariants() (smCounter.py:184-269): ';' + tags in the reference's order
int filter_string(std::string& f, uint32_t bits, const uint8_t* hp, int64_t i) {
    f = ";";
    if (!(bits & F_EVALUATED)) return SMC_ROWS_OK;
    if (bits & F_LM) f += "LM;";
    if (bits & F_LSM) f += "LSM;";
    if (bits & F_HPGATE) {                                                 // :195-203
        if (!hp || !(hp[i] & 128u)) return SMC_ROWS_E_HP;
        if (hp[i] & 1u) f += "HP;";
        if (hp[i] & 2u) f += "LowC;";
    }
    if (bits & F_DP) f += "DP;";
    if (bits & F_SB) f += "SB;";
    if (bits & F_LOWQ) f += "LowQ;";
    if (bits & F_R1CP) f += "R1CP;";
    if (bits & F_R2CP) f += "R2CP;";
    if (bits & F_PRIMERCP) f += "PrimerCP;";
    return SMC_ROWS_OK;
}

static const char FIXED_NAMES[5][4] = {"A", "C", "DEL", "T", "G"};
static const size_t FIXED_LEN[5] = {1, 1, 3, 1, 1};

int allele_name(const smc_rows_in& in, int32_t a, const char*& s, size_t& n) {
    if (a >= 0 && a < SMC_NFIXED) { s = FIXED_NAMES[a]; n = FIXED_LEN[a]; return SMC_ROWS_OK; }
    const int64_t j = (int64_t)a - SMC_NFIXED;
    if (j < 0 || j >= in.n_dyn || !in.dyn_names || !in.dyn_name_off) return SMC_ROWS_E_NAME;
    s = in.dyn_names + in.dyn_name_off[j]; n = (size_t)(in.dyn_name_off[j + 1] - in.dyn_name_off[j]);
    return n ? SMC_ROWS_OK : SMC_ROWS_E_NAME;
}

void emit_range(const Ctx& C, int64_t r0, int64_t r1, Chunk& out) {
    const smc_rows_in& in = *C.in;
    const size_t nl = (size_t)in.n_loci;
    auto LOC = [&](int f, int64_t i) { return in.loc[(size_t)f * nl + (size_t)i]; };
    auto CNT = [&](int a, int c, int64_t i) { return in.cnt[((size_t)a * SMC_NCNT + (size_t)c) * nl + (size_t)i]; };
    static const int ATGC[4] = {SMC_A_A, SMC_A_T, SMC_A_G, SMC_A_C};
    std::string fltr, fltr2, altbuf, typebuf;
    out.all.reserve((size_t)(r1 - r0) * 220);
    out.all_len.reserve((size_t)(r1 - r0));
    for (int64_t r = r0; r < r1; ++r) {
        const int64_t i = in.order ? in.order[r] : r;
        const size_t a0 = out.all.size(), c0 = out.cut.size(), v0 = out.vcf.size();
        auto fail = [&](int code, uint32_t st) { out.status = code; out.bad_row = r; out.bad_status = st; };
        if (i < 0 || i >= in.n_loci || in.ref_id[i] < 0 || in.ref_id[i] >= in.n_chroms) { fail(SMC_ROWS_E_ARG, 0); return; }
        const char* chrom = in.chroms[in.ref_id[i]];
        const int64_t pos = (int64_t)in.pos0[i] + 1;
        const char origRef[2] = {(char)in.ref_base[i], 0};
        const uint32_t status = (uint32_t)LOC(SMC_L_STATUS, i);
        if (status & (SMC_ST_NEED_DOWNSAMPLE | SMC_ST_UMI_OVERFLOW | SMC_ST_BAD_MASK)) { fail(SMC_ROWS_E_STATUS, status); return; }
        std::string& o = out.all;
        o += chrom; o.push_back('\t'); put_int(o, pos); o.push_back('\t'); o.push_back(origRef[0]);
        if (status & SMC_ST_ZERO_COVERAGE) {                                  // smCounter.py:492-494: 3 fields + 41 blanks + tag
            o.append(42, '\t'); o += "Zero_Coverage\n";
            out.all_len.push_back((int64_t)(o.size() - a0)); out.cut_len.push_back(0); out.vcf_len.push_back(0);
            continue;
        }
        o.resize(a0);                                                         // REF may change (indel): start the row again below
        const int64_t cvg = LOC(SMC_L_CVG, i), usedMT = LOC(SMC_L_USEDMT, i);
        int32_t alt_ref = in.alt_allele[i];
        const char* nm; size_t nn;
        int rc = allele_name(in, alt_ref, nm, nn);
        if (rc) { fail(rc, status); return; }
        Allele A = convert_to_vcf(origRef, nm, nn);
        rc = filter_string(fltr, in.fl1[i], in.hp1, i);
        if (rc) { fail(rc, status); return; }
        const char* ref = A.ref; size_t ref_n = A.ref_n;
        const char* alt = A.alt; size_t alt_n = A.alt_n;
        const char* vtype = A.vtype;
        if (in.biallelic[i]) {                                                 // smCounter.py:555-573
            const int32_t a2 = in.second_allele[i];
            const char* nm2; size_t nn2;
            rc = allele_name(in, a2, nm2, nn2);
            if (rc) { fail(rc, status); return; }
            const Allele B = convert_to_vcf(origRef, nm2, nn2);
            rc = filter_string(fltr2, in.fl2[i], in.hp2, i);
            if (rc) { fail(rc, status); return; }
            if (fltr == ";" && fltr2 == ";") {
                altbuf.assign(alt, alt_n); altbuf.push_back(','); altbuf.append(B.alt, B.alt_n);
                typebuf = lower_type(vtype); typebuf.push_back(','); typebuf += lower_type(B.vtype);
                alt = altbuf.data(); alt_n = altbuf.size(); vtype = typebuf.c_str();
            } else if (fltr != ";" && fltr2 == ";") {
                alt = B.alt; alt_n = B.alt_n; fltr = fltr2; alt_ref = a2;
            }
        }
        int64_t v_dp, v_mt, v_sm; double v_pi;
        if (alt_ref < SMC_NFIXED) {
            v_dp = CNT(alt_ref, SMC_C_ALLELE, i); v_mt = CNT(alt_ref, SMC_C_MT, i); v_sm = CNT(alt_ref, SMC_C_STRONG, i);
            v_pi = in.pi[(size_t)alt_ref * nl + (size_t)i];
        } else {
            const int64_t j = (int64_t)alt_ref - SMC_NFIXED;
            v_dp = in.dyn_cnt[j * SMC_NCNT + SMC_C_ALLELE]; v_mt = in.dyn_cnt[j * SMC_NCNT + SMC_C_MT]; v_sm = in.dyn_cnt[j * SMC_NCNT + SMC_C_STRONG];
            v_pi = in.dyn_pi[j];
        }
        const uint64_t k_pi = round_scaled(v_pi, 100), k_vaf = frac4(v_dp, cvg), k_vmf = frac4(v_mt, usedMT);
        const bool alt_is_del_word = alt_n == 3 && std::memcmp(alt, "DEL", 3) == 0;
        // ---- FILTER: main()'s repeat filters and the final form (smCounter.py:751-785)
        if (in.finalize) {
            if (k_pi / 100 >= 5 && !alt_is_del_word) {
                if (C.trf.first_hit(in.ref_id[i], pos) >= 0) fltr += "RepT;";       // (the VMF < 40 guard of :772 is always true)
                const int64_t h = C.rm.first_hit(in.ref_id[i], pos);
                if (h >= 0) fltr.append(in.rm_tags + in.rm_tag_off[h], (size_t)(in.rm_tag_off[h + 1] - in.rm_tag_off[h]));
            }
            if (fltr == ";") fltr = "PASS";
            else {
                size_t b = 0, e = fltr.size();
                while (b < e && fltr[b] == ';') ++b;
                while (e > b && fltr[e - 1] == ';') --e;
                fltr = fltr.substr(b, e - b);
            }
        }
        // ---- the 45 columns (smCounter.py:575-600)
        const size_t pi_at = [&]() {
            o += chrom; o.push_back('\t'); put_int(o, pos); o.push_back('\t'); o.append(ref, ref_n); o.push_back('\t');
            o.append(alt, alt_n); o.push_back('\t'); o += vtype; o.push_back('\t');
            put_int(o, cvg); o.push_back('\t'); put_int(o, LOC(SMC_L_ALLFRAG, i)); o.push_back('\t'); put_int(o, LOC(SMC_L_ALLMT, i)); o.push_back('\t');
            put_int(o, LOC(SMC_L_USEDFRAG, i)); o.push_back('\t'); put_int(o, usedMT); o.push_back('\t');
            return o.size();
        }();
        put_scaled(o, k_pi, 2);
        const size_t pi_len = o.size() - pi_at;
        o.push_back('\t'); put_int(o, v_dp); o.push_back('\t'); put_scaled(o, k_vaf, 4); o.push_back('\t'); put_int(o, v_mt); o.push_back('\t');
        const size_t vmf_at = o.size();
        put_scaled(o, k_vmf, 4);
        const size_t vmf_len = o.size() - vmf_at;
        o.push_back('\t'); put_int(o, v_sm);
        for (int k = 0; k < 4; ++k) { o.push_back('\t'); put_int(o, CNT(ATGC[k], SMC_C_ALLELE, i)); }
        for (int k = 0; k < 4; ++k) { o.push_back('\t'); put_scaled(o, frac4(CNT(ATGC[k], SMC_C_ALLELE, i), cvg), 4); }
        o.push_back('\t'); put_int(o, LOC(SMC_L_MT3, i)); o.push_back('\t'); put_int(o, LOC(SMC_L_MT5, i));
        o.push_back('\t'); put_int(o, LOC(SMC_L_MT7, i)); o.push_back('\t'); put_int(o, LOC(SMC_L_MT10, i));
        for (int k = 0; k < 4; ++k) { o.push_back('\t'); put_int(o, CNT(ATGC[k], SMC_C_MT, i)); }
        for (int k = 0; k < 4; ++k) { o.push_back('\t'); put_scaled(o, frac4(CNT(ATGC[k], SMC_C_MT, i), usedMT), 4); }
        for (int k = 0; k < 4; ++k) { o.push_back('\t'); put_int(o, CNT(ATGC[k], SMC_C_STRONG, i)); }
        for (int k = 0; k < 4; ++k) { o.push_back('\t'); put_scaled(o, round_scaled(in.pi[(size_t)ATGC[k] * nl + (size_t)i], 100), 2); }
        o.push_back('\t'); o += fltr; o.push_back('\n');
        out.all_len.push_back((int64_t)(o.size() - a0));
        // ---- called variants (smCounter.py:840-891)
        if (in.finalize && (int64_t)(k_pi / 100) >= (int64_t)in.threshold && !alt_is_del_word) {
            const std::string PI(o, pi_at, pi_len), VMF(o, vmf_at, vmf_len);
            const bool two = std::memchr(alt, ',', alt_n) != nullptr;
            const char* gt = two ? "1/2" : (!std::strcmp(chrom, "chrY") || !std::strcmp(chrom, "chrM")) ? "1" : k_vmf > 9500 ? "1/1" : "0/1";
            std::string& v = out.vcf;
            v += chrom; v.push_back('\t'); put_int(v, pos); v += "\t.\t"; v.append(ref, ref_n); v.push_back('\t'); v.append(alt, alt_n); v.push_back('\t');
            put_uint(v, k_pi / 100); v.push_back('\t'); v += fltr; v += "\tTYPE="; v += vtype; v += ";DP="; put_int(v, cvg); v += ";MT=";
            put_int(v, LOC(SMC_L_ALLMT, i)); v += ";UMT="; put_int(v, usedMT); v += ";PI="; v += PI; v += ";THR="; put_int(v, in.threshold);
            v += ";VMT="; put_int(v, v_mt); v += ";VMF="; v += VMF; v += ";VSM="; put_int(v, v_sm); v += "\tGT:AD:VF\t"; v += gt; v.push_back(':');
            put_int(v, usedMT - v_mt); v.push_back(','); put_int(v, v_mt); if (two) v += ",1";
            v.push_back(':'); v += VMF; v.push_back('\n');
            std::string& c = out.cut;
            c += chrom; c.push_back('\t'); put_int(c, pos); c.push_back('\t'); c.append(ref, ref_n); c.push_back('\t'); c.append(alt, alt_n); c.push_back('\t');
            c += vtype; c.push_back('\t'); put_int(c, cvg); c.push_back('\t'); put_int(c, LOC(SMC_L_ALLMT, i)); c.push_back('\t'); put_int(c, usedMT);
            c.push_back('\t'); c += PI; c.push_back('\t'); put_int(c, in.threshold); c.push_back('\t'); put_int(c, v_mt); c.push_back('\t'); c += VMF;
            c.push_back('\t'); put_int(c, v_sm); c.push_back('\t'); c += fltr; c.push_back('\n');
        }
        out.cut_len.push_back((int64_t)(out.cut.size() - c0)); out.vcf_len.push_back((int64_t)(out.vcf.size() - v0));
    }
}

}  // namespace

extern "C" int smc_rows_emit(const smc_rows_in* in, smc_rows_out* out) {
    if (!in || !out) return SMC_ROWS_E_ARG;
    std::memset(out, 0, sizeof *out);
    out->bad_row = -1;
    if (in->n_rows < 0 || in->n_loci < 0 || (in->n_rows > 0 && (!in->ref_id || !in->pos0 || !in->ref_base || !in->chroms || !in->loc || !in->cnt ||
                                                                 !in->pi || !in->alt_allele || !in->second_allele || !in->fl1 || !in->fl2 || !in->biallelic)))
        return SMC_ROWS_E_ARG;
    Ctx C; C.in = in;
    if (in->finalize) {
        if ((in->n_trf > 0 && (!in->trf_chrom || !in->trf_lo || !in->trf_hi)) ||
            (in->n_rm > 0 && (!in->rm_chrom || !in->rm_lo || !in->rm_hi || !in->rm_tags || !in->rm_tag_off))) return SMC_ROWS_E_ARG;
        C.trf.build(in->n_chroms, in->n_trf, in->trf_chrom, in->trf_lo, in->trf_hi);
        C.rm.build(in->n_chroms, in->n_rm, in->rm_chrom, in->rm_lo, in->rm_hi);
    }
    const int T = (int)std::min<int64_t>(smc_host::n_threads(in->threads), std::max<int64_t>(1, in->n_rows / 2048));
    std::vector<Chunk> chunks((size_t)T);
    smc_host::for_ranges((size_t)in->n_rows, T, [&](size_t r0, size_t r1, int t) { emit_range(C, (int64_t)r0, (int64_t)r1, chunks[(size_t)t]); });
    for (const Chunk& c : chunks)
        if (c.status != SMC_ROWS_OK) { out->bad_row = c.bad_row; out->bad_status = c.bad_status; return c.status; }
    auto gather = [&](std::string Chunk::*buf, std::vector<int64_t> Chunk::*lens, char*& dst, int64_t*& off) -> bool {
        size_t total = 0;
        for (const Chunk& c : chunks) total += (c.*buf).size();
        dst = (char*)std::malloc(total + 1);
        off = (int64_t*)std::malloc((size_t)(in->n_rows + 1) * sizeof(int64_t));
        if (!dst || !off) return false;
        size_t p = 0; int64_t r = 0; int64_t acc = 0;
        for (const Chunk& c : chunks) {
            std::memcpy(dst + p, (c.*buf).data(), (c.*buf).size()); p += (c.*buf).size();
            for (int64_t l : c.*lens) { off[r++] = acc; acc += l; }
        }
        off[r] = acc; dst[total] = 0;
        return r == in->n_rows;
    };
    bool ok = gather(&Chunk::all, &Chunk::all_len, out->all, out->all_off);
    ok = ok && gather(&Chunk::cut, &Chunk::cut_len, out->cut, out->cut_off);
    ok = ok && gather(&Chunk::vcf, &Chunk::vcf_len, out->vcf, out->vcf_off);
    if (!ok) { smc_rows_free(out); return SMC_ROWS_E_MEM; }
    return SMC_ROWS_OK;
}

extern "C" void smc_rows_free(smc_rows_out* out) {
    if (!out) return;
    std::free(out->all); std::free(out->all_off); std::free(out->cut); std::free(out->cut_off); std::free(out->vcf); std::free(out->vcf_off);
    out->all = out->cut = out->vcf = nullptr; out->all_off = out->cut_off = out->vcf_off = nullptr;
}
