// libsmc_bamio.so -- BAM (BGZF) -> flat SoA read buffers (include/smc_bamio.h).  Host-side input decoding only.
// Container format restated from the SAM/BAM specification (SAMv1 sections 4.1-4.2, the .bai index 5.2); zlib does the inflating.
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <array>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/smc_bamio.h"
#include "smc_host.h"
#include "smc_inflate.h"

using smc_host::for_each_thread;
using smc_host::for_ranges;

namespace {
thread_local std::string g_open_error;

// SMC_BAM_TIMING=1: per-phase wall clock on stderr (tuning aid)
smc_host::PhaseTimer phase_timer() { return smc_host::PhaseTimer("SMC_BAM_TIMING", "smc_bamio"); }

int out_of_memory(std::string& err, const char* what) { err = std::string("out of memory for ") + what; return -1; }

inline uint16_t rd16(const uint8_t* p) { uint16_t v; memcpy(&v, p, 2); return v; }
inline uint32_t rd32(const uint8_t* p) { uint32_t v; memcpy(&v, p, 4); return v; }
inline int32_t rdi32(const uint8_t* p) { int32_t v; memcpy(&v, p, 4); return v; }

// one BGZF block: its deflate payload at coff, and the bytes [lo, hi) of its isize inflated ones that go to uoff of the stream
struct Block { size_t coff, clen; size_t uoff; uint32_t isize, lo, hi; };

// .bai contents of one reference (SAMv1 5.2): chunks per bin (virtual offsets, [beg, end)) and the 16 kbp linear index
struct BaiChunk { uint64_t beg, end; };
struct BaiRef {
    std::unordered_map<uint32_t, std::vector<BaiChunk>> bins;
    std::vector<uint64_t> linear;
};

// malloc'ed and NOT zero-filled (std::vector::resize would touch every page once more, serially); false when out of memory.
// `slack` zeroed elements follow the `count` ones (the block decoder reads its input eight bytes at a time).
template <class T> struct Buf {
    T* p = nullptr; size_t n = 0;
    Buf() = default;
    Buf(const Buf&) = delete;
    Buf& operator=(const Buf&) = delete;
    ~Buf() { free(p); }
    bool resize(size_t count, size_t slack = 0) {
        free(p);
        p = (T*)malloc((count + slack ? count + slack : 1) * sizeof(T));
        n = p ? count : 0;
        if (p && slack) memset(p + count, 0, slack * sizeof(T));
        return p != nullptr;
    }
    size_t size() const { return n; }
    T* data() { return p; }
    const T* data() const { return p; }
    T& operator[](size_t i) { return p[i]; }
    const T& operator[](size_t i) const { return p[i]; }
};
}  // namespace

struct smc_bam {
    std::string err;
    Buf<uint8_t> raw;                         // inflated stream
    std::vector<std::string> ref_names;
    std::vector<int64_t> ref_lens;
    size_t first_record = 0;
    int threads = 1;
    // decoded buffers
    Buf<int32_t> ref_id, pos, nm, l_seq;
    Buf<uint16_t> flag, n_cigar;
    Buf<uint8_t> mapq, seq, qual;
    Buf<int64_t> seq_off, qual_off, cigar_off;
    Buf<uint64_t> umi;
    Buf<uint32_t> frag_id, cigar;
    std::vector<std::string> dict_umis;
    Buf<int32_t> store_lo, store_len;           // stored window per read (trim mode)
    uint64_t qual_hist[256] = {0};              // how often every phred value occurs among the stored qualities
    int trim = 0;
    bool decoded = false;
    // opened through an index (smc_bam_open_indexed): raw holds only the header until smc_bam_decode reads the chunks it needs
    bool indexed = false;
    std::string path, index_path;
    size_t file_size = 0;
    std::vector<BaiRef> bai;
};

// the BGZF header at seg[off] (seg has n bytes): 0 and its BSIZE (the block's size - 1, from the BC subfield) and XLEN;
// 1 not a BGZF header, 2 no BC subfield inside the n bytes
static int bgzf_header(const uint8_t* seg, size_t n, size_t off, size_t& bsize, size_t& xlen) {
    if (off + 18 > n || seg[off] != 0x1f || seg[off + 1] != 0x8b || seg[off + 2] != 8 || !(seg[off + 3] & 4)) return 1;
    xlen = rd16(&seg[off + 10]);
    size_t p = off + 12, end = p + xlen;
    int64_t bs = -1;
    while (p + 4 <= end && end <= n) {
        const uint16_t slen = rd16(&seg[p + 2]);
        if (seg[p] == 66 && seg[p + 1] == 67 && slen == 2) bs = rd16(&seg[p + 4]);
        p += 4 + slen;
    }
    if (bs < 0) return 2;
    bsize = (size_t)bs;
    return 0;
}

// the BGZF block at seg[off] (seg has n bytes): 0 and the block (coff relative to seg) and the offset of the next one;
// 1 not a BGZF block, 2 truncated or malformed
static int bgzf_block(const uint8_t* seg, size_t n, size_t off, Block& b, size_t& next) {
    size_t bsize = 0, xlen = 0;
    const int rc = bgzf_header(seg, n, off, bsize, xlen);
    if (rc != 0) return rc;
    if (off + bsize + 1 > n || bsize + 1 < 12 + xlen + 8) return 2;
    b.coff = off + 12 + xlen;
    b.clen = (size_t)bsize + 1 - 12 - xlen - 8;
    b.isize = rd32(&seg[off + bsize + 1 - 4]);
    b.lo = 0; b.hi = b.isize;
    next = off + (size_t)bsize + 1;
    return 0;
}

// inflate every block of src (which is readable 64 bytes past its last block) and store its bytes [lo, hi) at out[uoff];
// a block cut by a chunk boundary is inflated into a scratch buffer first
static int inflate_blocks(const uint8_t* src, const std::vector<Block>& blocks, int threads, Buf<uint8_t>& out, std::string& err) {
    std::atomic<size_t> next(0);
    std::atomic<int> bad(0);
    // the blocks go through the decoder of smc_inflate.h; a block it rejects is given to zlib (SMC_INFLATE=zlib: zlib for all)
    static const bool own_inflate = [] { const char* ev = getenv("SMC_INFLATE"); return !(ev && strcmp(ev, "zlib") == 0); }();
    auto work = [&](int) {
        z_stream zs;
        std::vector<uint8_t> scratch;
        for (;;) {
            const size_t i = next.fetch_add(1);
            if (i >= blocks.size() || bad.load()) break;
            const Block& b = blocks[i];
            if (b.hi == b.lo) continue;
            const bool whole = b.lo == 0 && b.hi == b.isize;
            if (!whole && scratch.size() < b.isize) scratch.resize(b.isize);
            uint8_t* dst = whole ? &out[b.uoff] : scratch.data();
            if (!(own_inflate && smc_inflate_raw(&src[b.coff], b.clen, dst, b.isize) == 0)) {
                memset(&zs, 0, sizeof(zs));
                if (inflateInit2(&zs, -15) != Z_OK) { bad = 1; break; }
                zs.next_in = const_cast<Bytef*>(&src[b.coff]); zs.avail_in = (uInt)b.clen;
                zs.next_out = dst; zs.avail_out = b.isize;
                const int rc = inflate(&zs, Z_FINISH);
                inflateEnd(&zs);
                if (rc != Z_STREAM_END || zs.avail_out != 0) { bad = 1; break; }
            }
            if (!whole) memcpy(&out[b.uoff], dst + b.lo, b.hi - b.lo);
        }
    };
    for_each_thread(std::max(1, std::min<int>(threads, (int)blocks.size())), work);
    if (bad.load()) { err = "zlib inflate failed on a BGZF block"; return -1; }
    return 0;
}

static int inflate_all(const Buf<uint8_t>& file, int threads, Buf<uint8_t>& out, std::string& err) {
    std::vector<Block> blocks;
    size_t off = 0, uoff = 0;
    const size_t n = file.size();
    while (off < n) {
        Block b;
        size_t nxt = 0;
        const int rc = bgzf_block(file.data(), n, off, b, nxt);
        if (rc == 1) { err = "not a BGZF block at offset " + std::to_string(off); return -1; }
        if (rc == 2) { err = "truncated or malformed BGZF block at offset " + std::to_string(off); return -1; }
        b.uoff = uoff;
        uoff += b.isize;
        blocks.push_back(b);
        off = nxt;
    }
    if (!out.resize(uoff)) return out_of_memory(err, "the inflated BAM");
    return inflate_blocks(file.data(), blocks, threads, out, err);
}

// pread the pieces (file offset, buffer offset, length) on up to `threads` threads; false on a short read
static bool pread_pieces(int fd, uint8_t* buf, const std::vector<std::array<size_t, 3>>& pieces, int threads) {
    std::atomic<size_t> next(0);
    std::atomic<int> short_read(0);
    auto rd = [&](int) {
        for (size_t i; (i = next.fetch_add(1)) < pieces.size() && !short_read.load();) {
            size_t a = 0;
            const size_t off = pieces[i][0], len = pieces[i][2];
            uint8_t* dst = buf + pieces[i][1];
            while (a < len) {
                const ssize_t k = pread(fd, dst + a, len - a, (off_t)(off + a));
                if (k <= 0) { short_read = 1; return; }
                a += (size_t)k;
            }
        }
    };
    for_each_thread((int)std::max<size_t>(1, std::min<size_t>((size_t)threads, pieces.size())), rd);
    return !short_read.load();
}

// [off, off + len) of the file cut into pieces of at most 4 MiB, stored from buf_off on
static void add_pieces(std::vector<std::array<size_t, 3>>& pieces, size_t off, size_t buf_off, size_t len) {
    const size_t piece = size_t(4) << 20;
    for (size_t a = 0; a < len; a += piece) pieces.push_back({off + a, buf_off + a, std::min(piece, len - a)});
}

// the whole file (usually in the page cache) read by all threads, each its own ranges (pread), plus 64 zero bytes of slack:
// the block decoder reads its input eight bytes at a time
static int read_whole_file(const char* path, int threads, Buf<uint8_t>& file, std::string& err) {
    const int fd = open(path, O_RDONLY);
    if (fd < 0) { err = std::string("smc_bam_open: cannot open ") + path; return -1; }
    struct stat st;
    const size_t sz = fstat(fd, &st) == 0 && st.st_size > 0 ? (size_t)st.st_size : 0;
    if (!file.resize(sz, 64)) { close(fd); err = "smc_bam_open: out of memory"; return -1; }
    std::vector<std::array<size_t, 3>> pieces;
    add_pieces(pieces, 0, 0, sz);
    const bool ok = pread_pieces(fd, file.p, pieces, threads);
    close(fd);
    if (!ok) { err = "smc_bam_open: short read"; return -1; }
    return 0;
}

// magic, header text and reference list from the start of the inflated stream: 0 (h->ref_names / ref_lens / first_record set),
// 1 the stream ends before the reference list does (err says how), -1 not a BAM stream
static int parse_header(const uint8_t* r, size_t n, smc_bam* h, std::string& err) {
    h->ref_names.clear(); h->ref_lens.clear();
    if (n >= 4 && memcmp(r, "BAM\1", 4) != 0) { err = "not a BAM file (bad magic)"; return -1; }
    if (n < 12) { err = "not a BAM file (bad magic)"; return 1; }
    const int32_t l_text = rdi32(&r[4]);
    if (l_text < 0) { err = "truncated BAM header"; return -1; }
    size_t p = 8 + (size_t)l_text;
    if (p + 4 > n) { err = "truncated BAM header"; return 1; }
    const int32_t n_ref = rdi32(&r[p]);
    p += 4;
    for (int32_t i = 0; i < n_ref; ++i) {
        if (p + 4 > n) { err = "truncated BAM reference list"; return 1; }
        const int32_t l_name = rdi32(&r[p]);
        if (l_name < 1) { err = "truncated BAM reference list"; return -1; }
        if (p + 8 + (size_t)l_name > n) { err = "truncated BAM reference list"; return 1; }
        h->ref_names.emplace_back(reinterpret_cast<const char*>(&r[p + 4]), (size_t)l_name - 1);
        h->ref_lens.push_back(rdi32(&r[p + 4 + l_name]));
        p += 8 + (size_t)l_name;
    }
    h->first_record = p;
    return 0;
}

static void timing_bytes(const char* what, size_t compressed, size_t inflated) {
    if (getenv("SMC_BAM_TIMING")) fprintf(stderr, "[smc_bamio] %s: compressed bytes read %zu, inflated bytes %zu\n", what, compressed, inflated);
}

extern "C" int smc_bam_open(const char* path, int threads, smc_bam** out) {
    if (!path || !out) { g_open_error = "smc_bam_open: null argument"; return -2; }
    auto pt = phase_timer();
    threads = smc_host::n_threads(threads);
    Buf<uint8_t> file;
    if (read_whole_file(path, threads, file, g_open_error) != 0) return -1;
    pt.lap("read file");
    smc_bam* h = new smc_bam();
    h->threads = threads;
    if (inflate_all(file, threads, h->raw, g_open_error) != 0) { delete h; return -1; }
    pt.lap("inflate");
    timing_bytes("whole file", file.size(), h->raw.size());
    if (parse_header(h->raw.data(), h->raw.size(), h, g_open_error) != 0) { delete h; return -1; }
    *out = h;
    return 0;
}

// ------------------------------------------------------------------------------------------------------------
// Region access through a .bai (SAMv1 5.2)
// ------------------------------------------------------------------------------------------------------------
static int parse_bai(const std::string& ipath, size_t n_ref_bam, std::vector<BaiRef>& refs, std::string& err) {
    const std::string who = "BAM index " + ipath + ": ";
    FILE* fh = fopen(ipath.c_str(), "rb");
    if (!fh) { err = who + "cannot open"; return -3; }
    std::vector<uint8_t> d;
    uint8_t buf[1 << 16];
    for (size_t k; (k = fread(buf, 1, sizeof(buf), fh)) > 0;) d.insert(d.end(), buf, buf + k);
    fclose(fh);
    const size_t n = d.size();
    size_t p = 0;
    auto truncated = [&]() { err = who + "truncated or malformed at byte " + std::to_string(p); return -3; };
    if (n < 8 || memcmp(d.data(), "BAI\1", 4) != 0) { err = who + "bad magic (not a .bai file)"; return -3; }
    const int32_t n_ref = rdi32(&d[4]);
    p = 8;
    if (n_ref < 0 || (size_t)n_ref != n_ref_bam) {
        err = who + "n_ref is " + std::to_string(n_ref) + " but the BAM header has " + std::to_string(n_ref_bam) + " references";
        return -3;
    }
    refs.assign((size_t)n_ref, BaiRef());
    for (int32_t r = 0; r < n_ref; ++r) {
        if (p + 4 > n) return truncated();
        const int32_t n_bin = rdi32(&d[p]);
        p += 4;
        if (n_bin < 0) return truncated();
        for (int32_t k = 0; k < n_bin; ++k) {
            if (p + 8 > n) return truncated();
            const uint32_t bin = rd32(&d[p]);
            const int32_t n_chunk = rdi32(&d[p + 4]);
            p += 8;
            if (n_chunk < 0 || p + 16 * (size_t)n_chunk > n) return truncated();
            if (bin != 37450) {                          // 37450: the metadata pseudo-bin (reference span, mapped / unmapped counts)
                auto& v = refs[(size_t)r].bins[bin];
                for (int32_t c = 0; c < n_chunk; ++c) {
                    BaiChunk ch;
                    memcpy(&ch.beg, &d[p + 16 * (size_t)c], 8); memcpy(&ch.end, &d[p + 16 * (size_t)c + 8], 8);
                    v.push_back(ch);
                }
            }
            p += 16 * (size_t)n_chunk;
        }
        if (p + 4 > n) return truncated();
        const int32_t n_intv = rdi32(&d[p]);
        p += 4;
        if (n_intv < 0 || p + 8 * (size_t)n_intv > n) return truncated();
        refs[(size_t)r].linear.resize((size_t)n_intv);
        if (n_intv) memcpy(refs[(size_t)r].linear.data(), &d[p], 8 * (size_t)n_intv);
        p += 8 * (size_t)n_intv;
    }
    if (p != n && p + 8 != n) return truncated();      // nothing, or the optional n_no_coor
    return 0;
}

extern "C" int smc_bam_open_indexed(const char* path, const char* index_path, int threads, smc_bam** out) {
    if (!path || !index_path || !out) { g_open_error = "smc_bam_open_indexed: null argument"; return -2; }
    auto pt = phase_timer();
    threads = smc_host::n_threads(threads);
    const int fd = open(path, O_RDONLY);
    if (fd < 0) { g_open_error = std::string("smc_bam_open: cannot open ") + path; return -1; }
    struct stat st;
    const size_t size = fstat(fd, &st) == 0 && st.st_size > 0 ? (size_t)st.st_size : 0;
    smc_bam* h = new smc_bam();
    h->threads = threads; h->indexed = true; h->path = path; h->index_path = index_path; h->file_size = size;
    // the header: BGZF blocks from offset 0, one at a time, until the header text and the reference list are complete
    std::vector<uint8_t> comp((size_t(1) << 16) + 64, 0), hdr;
    size_t off = 0, comp_read = 0;
    int st_hdr = 1;
    g_open_error = "not a BAM file (bad magic)";
    while (st_hdr == 1 && off < size) {
        const size_t len = std::min(size - off, size_t(1) << 16);           // a BGZF block is at most 64 KiB
        std::vector<std::array<size_t, 3>> piece{{off, 0, len}};
        if (!pread_pieces(fd, comp.data(), piece, 1)) { g_open_error = "smc_bam_open: short read"; break; }
        memset(comp.data() + len, 0, 64);
        Block b;
        size_t nxt = 0;
        const int rc = bgzf_block(comp.data(), len, 0, b, nxt);
        if (rc) { g_open_error = (rc == 1 ? "not a BGZF block at offset " : "truncated or malformed BGZF block at offset ") + std::to_string(off); st_hdr = -1; break; }
        comp_read += nxt;
        Buf<uint8_t> one;
        b.uoff = 0;
        if (!one.resize(b.isize)) { g_open_error = "smc_bam_open: out of memory"; st_hdr = -1; break; }
        if (inflate_blocks(comp.data(), std::vector<Block>{b}, 1, one, g_open_error) != 0) { st_hdr = -1; break; }
        hdr.insert(hdr.end(), one.data(), one.data() + b.isize);
        st_hdr = parse_header(hdr.data(), hdr.size(), h, g_open_error);
        off += nxt;
    }
    close(fd);
    if (st_hdr != 0) { delete h; return -1; }
    pt.lap("header blocks");
    timing_bytes("header", comp_read, hdr.size());
    const int rc = parse_bai(h->index_path, h->ref_names.size(), h->bai, g_open_error);
    if (rc != 0) { delete h; return rc; }
    pt.lap("index parse");
    *out = h;
    return 0;
}

// SAMv1 5.3: the bins that may hold a record overlapping [beg, end)
static void reg2bins(int64_t beg, int64_t end, std::vector<uint32_t>& out) {
    out.clear();
    --end;
    out.push_back(0);
    for (int64_t k = 1 + (beg >> 26); k <= 1 + (end >> 26); ++k) out.push_back((uint32_t)k);
    for (int64_t k = 9 + (beg >> 23); k <= 9 + (end >> 23); ++k) out.push_back((uint32_t)k);
    for (int64_t k = 73 + (beg >> 20); k <= 73 + (end >> 20); ++k) out.push_back((uint32_t)k);
    for (int64_t k = 585 + (beg >> 17); k <= 585 + (end >> 17); ++k) out.push_back((uint32_t)k);
    for (int64_t k = 4681 + (beg >> 14); k <= 4681 + (end >> 14); ++k) out.push_back((uint32_t)k);
}

// h->raw = the records of the index chunks that the intervals need, in file order.  A chunk [beg, end) covers whole records,
// so the concatenated slices are a valid record chain; chunks that share a BGZF block are merged, which adds only whole records
// in between (dropped by the interval filter like any other) and inflates every block once.
static int load_chunks(smc_bam* h, int64_t n_iv, const int32_t* iv_ref, const int32_t* iv_start, const int32_t* iv_end) {
    auto pt = phase_timer();
    const std::string who = "BAM index " + h->index_path + ": ";
    auto chunk_error = [&](const BaiChunk& c, const std::string& what) {
        h->err = who + "chunk [" + std::to_string(c.beg) + ", " + std::to_string(c.end) + ") " + what;
        return -3;
    };
    std::vector<BaiChunk> ch;
    std::vector<uint32_t> bins;
    for (int64_t k = 0; k < n_iv; ++k) {
        const int32_t rid = iv_ref[k];
        if (rid < 0 || (size_t)rid >= h->bai.size()) continue;
        const int64_t beg = std::max<int64_t>(0, iv_start[k]), end = std::min<int64_t>(iv_end[k], int64_t(1) << 29);
        if (end <= beg) continue;
        const BaiRef& R = h->bai[(size_t)rid];
        const uint64_t min_off = R.linear.empty() ? 0 : R.linear[std::min<size_t>((size_t)(beg >> 14), R.linear.size() - 1)];
        reg2bins(beg, end, bins);
        for (uint32_t bin : bins) {
            auto it = R.bins.find(bin);
            if (it == R.bins.end()) continue;
            for (const BaiChunk& c : it->second)
                if (c.end > min_off && c.end > c.beg) ch.push_back(c);
        }
    }
    std::sort(ch.begin(), ch.end(), [](const BaiChunk& a, const BaiChunk& b) { return a.beg < b.beg || (a.beg == b.beg && a.end < b.end); });
    std::vector<BaiChunk> merged;
    for (const BaiChunk& c : ch) {
        if (!merged.empty() && (c.beg >> 16) <= (merged.back().end >> 16)) merged.back().end = std::max(merged.back().end, c.end);
        else merged.push_back(c);
    }
    pt.lap("index: chunk query");
    // compressed byte range of every merged chunk: from the block of its start to the end of the block of its end (or to the start
    // of that block when the end is at its offset 0)
    const int fd = open(h->path.c_str(), O_RDONLY);
    if (fd < 0) { h->err = "smc_bam_decode: cannot open " + h->path; return -1; }
    struct Range { size_t cbeg, cend, buf; };
    std::vector<Range> ranges;
    size_t total = 0;
    int rc = 0;
    for (const BaiChunk& c : merged) {
        const size_t cbeg = (size_t)(c.beg >> 16), cend = (size_t)(c.end >> 16);
        size_t stop = cend;
        if (cbeg >= h->file_size || cend > h->file_size || (cend == h->file_size && (c.end & 0xffff))) {
            rc = chunk_error(c, "points past the end of " + h->path); break;
        }
        if (c.end & 0xffff) {                       // the block holding the chunk's end: its size from its own header
            uint8_t head[18 + 64];
            const size_t len = cend < h->file_size ? std::min<size_t>(sizeof(head), h->file_size - cend) : 0;
            std::vector<std::array<size_t, 3>> piece{{cend, 0, len}};
            size_t bsize = 0, xlen = 0;
            if (!pread_pieces(fd, head, piece, 1) || bgzf_header(head, len, 0, bsize, xlen) != 0) {
                h->err = who + "chunk end at virtual offset " + std::to_string(c.end) + " is not in a BGZF block of " + h->path;
                rc = -3; break;
            }
            stop = cend + bsize + 1;
        }
        if (stop > h->file_size || cbeg >= h->file_size) { rc = chunk_error(c, "points past the end of " + h->path); break; }
        if (cbeg >= stop) { rc = chunk_error(c, "is malformed"); break; }
        ranges.push_back({cbeg, stop, total});
        total += stop - cbeg;
    }
    Buf<uint8_t> comp;
    if (rc == 0 && !comp.resize(total, 64)) rc = out_of_memory(h->err, "the compressed chunks");
    if (rc == 0) {
        std::vector<std::array<size_t, 3>> pieces;
        for (const Range& g : ranges) add_pieces(pieces, g.cbeg, g.buf, g.cend - g.cbeg);
        if (!pread_pieces(fd, comp.p, pieces, h->threads)) { h->err = "smc_bam_decode: short read of " + h->path; rc = -1; }
    }
    close(fd);
    if (rc != 0) return rc;
    pt.lap("index: chunk reads");
    // the blocks of every range, each with the slice of its inflated bytes that the chunk covers
    std::vector<Block> blocks;
    size_t uoff = 0;
    for (size_t g = 0; g < ranges.size(); ++g) {
        const Range& R = ranges[g];
        const BaiChunk& c = merged[g];
        const uint8_t* seg = comp.p + R.buf;
        const size_t n = R.cend - R.cbeg;
        for (size_t off = 0; off < n;) {
            Block b;
            size_t nxt = 0;
            const bool last = bgzf_block(seg, n, off, b, nxt) == 0 && nxt == n;
            if (nxt == 0 || (last && (c.end & 0xffff) && off != (size_t)(c.end >> 16) - R.cbeg))
                return chunk_error(c, "does not point at BGZF blocks of " + h->path + " (offset " + std::to_string(R.cbeg + off) + ")");
            if (off == 0) b.lo = (uint32_t)(c.beg & 0xffff);
            if (last && (c.end & 0xffff)) b.hi = (uint32_t)(c.end & 0xffff);
            if (b.lo > b.hi || b.hi > b.isize) return chunk_error(c, "points past the data of a BGZF block of " + h->path);
            b.coff += R.buf;
            b.uoff = uoff;
            uoff += b.hi - b.lo;
            blocks.push_back(b);
            off = nxt;
        }
    }
    if (!h->raw.resize(uoff)) return out_of_memory(h->err, "the inflated chunks");
    if (inflate_blocks(comp.data(), blocks, h->threads, h->raw, h->err) != 0) return -1;
    h->first_record = 0;
    pt.lap("index: chunk inflate");
    timing_bytes("index chunks", total, uoff);
    return 0;
}

extern "C" void smc_bam_close(smc_bam* h) { delete h; }
extern "C" int smc_bam_inflate_raw(const uint8_t* in, int64_t in_len, uint8_t* out, int64_t out_len) {
    if (!in || !out || in_len < 0 || out_len < 0) return -2;
    return smc_inflate_raw(in, (size_t)in_len, out, (size_t)out_len);
}
extern "C" void smc_bam_set_trim(smc_bam* h, int trim) { if (h) h->trim = trim ? 1 : 0; }
extern "C" const char* smc_bam_last_error(smc_bam* h) { return h ? h->err.c_str() : g_open_error.c_str(); }
extern "C" int smc_bam_n_refs(smc_bam* h) { return h ? (int)h->ref_names.size() : 0; }
extern "C" const char* smc_bam_ref_name(smc_bam* h, int i) { return (h && i >= 0 && i < (int)h->ref_names.size()) ? h->ref_names[i].c_str() : ""; }
extern "C" int64_t smc_bam_ref_length(smc_bam* h, int i) { return (h && i >= 0 && i < (int)h->ref_lens.size()) ? h->ref_lens[i] : -1; }
extern "C" const char* smc_bam_dict_umi(smc_bam* h, int64_t i) { return (h && i >= 0 && i < (int64_t)h->dict_umis.size()) ? h->dict_umis[(size_t)i].c_str() : ""; }

// value of the first NM tag in [p, end), 0 when absent (smCounter.py:329-334)
static int32_t first_nm(const uint8_t* p, const uint8_t* end) {
    while (p + 3 <= end) {
        const uint8_t t0 = p[0], t1 = p[1], ty = p[2];
        p += 3;
        size_t sz = 0;
        switch (ty) {
            case 'A': case 'c': case 'C': sz = 1; break;
            case 's': case 'S': sz = 2; break;
            case 'i': case 'I': case 'f': sz = 4; break;
            case 'Z': case 'H': { const void* q = memchr(p, 0, (size_t)(end - p)); if (!q) return 0; p = (const uint8_t*)q + 1; continue; }
            case 'B': {
                if (p + 5 > end) return 0;
                const uint8_t sub = p[0];
                const int32_t cnt = rdi32(p + 1);
                const size_t es = (sub == 'c' || sub == 'C') ? 1 : (sub == 's' || sub == 'S') ? 2 : 4;
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

// ------------------------------------------------------------------------------------------------------------
// Record decode (smc_bam_decode), four passes, each a function below:
//   1 record_offsets   record boundaries (block_size chain: byte ranges walked in parallel, serial walk as the fallback);
//   2 record_fields    per record: fields, interval filter, barcode code, 128-bit hash of the (barcode, readid) identity;
//   3 fragment_firsts  the first record of every identity (hash partitions, every hit verified on the name bytes);
//     number_reads     output slots and payload offsets of the kept reads, fragment ids by first appearance, dictionary of
//                      non-ACGT / long barcodes;
//   4 copy_records     scalars and payloads copied to their final places, the histogram of the stored qualities.
// ------------------------------------------------------------------------------------------------------------
namespace {
struct RecInfo {
    uint32_t keep;                 // 1 kept, 0 dropped
    uint32_t store_lo, store_len;  // stored window of the bases / qualities (whole read unless trimming)
    uint32_t bc_off, bc_len;       // barcode bytes inside qname
    uint32_t rid_len;              // readid = qname[0, rid_len)
    uint64_t h1, h2;               // hash of (barcode, readid)
    uint64_t code;                 // packed barcode, 0 = needs the dictionary
};

inline uint64_t mix64(uint64_t x) { x ^= x >> 32; x *= 0xd6e8feb86659fd93ull; x ^= x >> 32; x *= 0xd6e8feb86659fd93ull; x ^= x >> 32; return x; }
inline void hash_bytes(const uint8_t* p, size_t n, uint64_t& a, uint64_t& b) {
    while (n >= 8) { uint64_t w; memcpy(&w, p, 8); a = mix64(a ^ w); b = (b + w) * 0x9e3779b97f4a7c15ull; b ^= b >> 29; p += 8; n -= 8; }
    uint64_t w = 0; memcpy(&w, p, n);
    a = mix64(a ^ w ^ ((uint64_t)n << 56)); b = (b + w + n) * 0x9e3779b97f4a7c15ull; b ^= b >> 29;
}

template <class F> void parallel_for(size_t n, int threads, F&& f) {       // f(begin, end, thread); one thread per 4096 items at most
    for_ranges(n, (int)std::max<size_t>(1, std::min<size_t>((size_t)threads, (n + 4095) / 4096)), f);
}

// The target intervals of every reference, sorted and merged where they overlap.  Intervals that only touch ([a, b) and
// [b, c)) stay apart: a read without reference length at b touches neither, and merging them would make it touch [a, c).
struct Targets {
    std::vector<std::vector<std::pair<int64_t, int64_t>>> by_ref;

    Targets(size_t nref, int64_t n_iv, const int32_t* iv_ref, const int32_t* iv_start, const int32_t* iv_end) : by_ref(nref) {
        for (int64_t k = 0; k < n_iv; ++k)
            if (iv_ref[k] >= 0 && (size_t)iv_ref[k] < nref && iv_end[k] > iv_start[k]) by_ref[(size_t)iv_ref[k]].push_back({iv_start[k], iv_end[k]});
        for (auto& v : by_ref) {
            std::sort(v.begin(), v.end());
            size_t m = 0;
            for (const auto& pr : v) {
                if (m > 0 && pr.first < v[m - 1].second) v[m - 1].second = std::max(v[m - 1].second, pr.second);
                else v[m++] = pr;
            }
            v.resize(m);
        }
    }
    // the intervals that the read [s, e) touches (start < e and end > s): [first, last), empty when the read touches no target.
    // Starts and ends both ascend, so each bound is one binary search.
    using It = std::vector<std::pair<int64_t, int64_t>>::const_iterator;
    std::pair<It, It> touched(int32_t rid, int64_t s, int64_t e) const {
        const auto& v = by_ref[(size_t)rid];
        return {std::partition_point(v.begin(), v.end(), [&](const std::pair<int64_t, int64_t>& iv) { return iv.second <= s; }),
                std::partition_point(v.begin(), v.end(), [&](const std::pair<int64_t, int64_t>& iv) { return iv.first < e; })};
    }
};
}  // namespace

// h->raw = the records to decode.  A handle opened through an index holds only the header so far: the records come from the
// index chunks the intervals need, or from the whole file when there are no intervals.
static int load_records(smc_bam* h, int64_t n_iv, const int32_t* iv_ref, const int32_t* iv_start, const int32_t* iv_end) {
    if (!h->indexed) return 0;
    h->indexed = false;
    if (n_iv > 0) return load_chunks(h, n_iv, iv_ref, iv_start, iv_end);
    auto pt = phase_timer();
    Buf<uint8_t> file;
    if (read_whole_file(h->path.c_str(), h->threads, file, h->err) != 0 || inflate_all(file, h->threads, h->raw, h->err) != 0) return -1;
    pt.lap("read + inflate whole file");
    timing_bytes("whole file", file.size(), h->raw.size());
    return 0;
}

// ---- pass 1: record boundaries.  The block_size chain is a serial pointer chase (one cache miss per record), so the stream
// is cut into byte ranges that are walked in parallel: a range that does not start the stream finds its first record by
// testing candidates for plausibility (three consistent records in a row), and the result is accepted only if every
// range's walk ends exactly where the next range started -- by induction from the known first record the chain is then
// the true one.  Anything else (including a malformed record) falls back to the plain serial walk and its error report.
static int record_offsets(const uint8_t* r, size_t begin, size_t size, size_t nref, int threads, std::vector<size_t>& offs, std::string& err) {
    auto plausible = [&](size_t p) -> size_t {                // 0 = no; else offset of the next record
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
    };
    const size_t span = size > begin ? size - begin : 0;
    const int T = (int)std::max<size_t>(1, std::min<size_t>((size_t)threads, span / (4u << 20)));
    bool ok = T > 1;
    if (ok) {
        std::vector<std::vector<size_t>> part(T);
        std::vector<size_t> first(T, SIZE_MAX), last(T, SIZE_MAX);
        std::vector<char> good(T, 1);
        for_each_thread(T, [&](int t) {
            const size_t lo = begin + span * (size_t)t / T, hi = t + 1 == T ? size : begin + span * (size_t)(t + 1) / T;
            size_t p = lo;
            if (t > 0) {                                         // first plausible chain of three at or after lo
                for (;; ++p) {
                    if (p + 4 > hi + (1u << 20) || p + 4 > size) { good[t] = 0; return; }
                    size_t q = plausible(p);
                    if (!q) continue;
                    size_t q2 = q + 4 <= size ? plausible(q) : (q == size ? q : 0);
                    if (!q2) continue;
                    if (q2 != size && q2 + 4 <= size && !plausible(q2)) continue;
                    break;
                }
            }
            first[t] = p;
            part[t].reserve((hi - lo) / 200 + 16);
            while (p + 4 <= size && p < hi) {
                const int32_t bs = rdi32(&r[p]);
                if (bs < 32 || p + 4 + (size_t)bs > size) { good[t] = 0; return; }
                part[t].push_back(p);
                p += 4 + (size_t)bs;
            }
            last[t] = p;
        });
        for (int t = 0; t < T && ok; ++t) ok = good[t] && (t + 1 == T || last[t] == first[t + 1]);
        if (ok && last[T - 1] + 4 <= size) ok = false;          // trailing bytes that are not a record: let the serial walk judge
        if (ok) {
            size_t tot = 0;
            for (auto& v : part) tot += v.size();
            offs.reserve(tot);
            for (auto& v : part) offs.insert(offs.end(), v.begin(), v.end());
        }
    }
    if (!ok) {
        offs.reserve(size / 200 + 16);
        for (size_t p = begin; p + 4 <= size;) {
            const int32_t bs = rdi32(&r[p]);
            if (bs < 32 || p + 4 + (size_t)bs > size) { err = "truncated BAM record at offset " + std::to_string(p); return -1; }
            offs.push_back(p);
            p += 4 + (size_t)bs;
        }
    }
    return 0;
}

// ---- pass 2: per record the fields, the interval filter (tg: null without intervals), the stored window (trim), the barcode
// code and the identity hash; n_kept = the reads kept
static int record_fields(const uint8_t* r, const std::vector<size_t>& offs, size_t nref, const Targets* tg, bool trim, int threads,
                         Buf<RecInfo>& info, size_t& n_kept, std::string& err) {
    const size_t nrec = offs.size();
    if (!info.resize(nrec)) return out_of_memory(err, "the record table");   // pass 2 writes keep for every record, the rest for kept ones
    std::atomic<size_t> bad_rec(SIZE_MAX);
    std::atomic<size_t> kept(0);
    parallel_for(nrec, threads, [&](size_t a, size_t e, int) {
        size_t kept_here = 0;
        struct AddKept { std::atomic<size_t>& tot; size_t& k; ~AddKept() { tot += k; } } add_kept{kept, kept_here};
        for (size_t i = a; i < e; ++i) {
            RecInfo& R = info[i];
            R.keep = 0;
            const uint8_t* b = &r[offs[i] + 4];
            const int32_t bs = rdi32(&r[offs[i]]);
            const uint8_t* rec_end = b + bs;
            const int32_t refID = rdi32(b), pos = rdi32(b + 4);
            const uint8_t l_rn = b[8];
            const uint16_t n_cig = rd16(b + 12), flag = rd16(b + 14);
            const int32_t l_seq = rdi32(b + 16);
            const char* qname = reinterpret_cast<const char*>(b + 32);
            const uint8_t* cig = b + 32 + l_rn;
            const uint8_t* sq = cig + 4 * (size_t)n_cig;
            const uint8_t* ql = sq + ((size_t)(l_seq < 0 ? 0 : l_seq) + 1) / 2;
            if (l_seq < 0 || ql + l_seq > rec_end) {
                size_t cur = bad_rec.load();
                while (i < cur && !bad_rec.compare_exchange_weak(cur, i)) {}
                continue;
            }
            if ((flag & 0x4) || refID < 0 || (size_t)refID >= nref) continue;
            R.store_lo = 0; R.store_len = (uint32_t)l_seq;
            if (tg) {
                int64_t reflen = 0;
                int n_run = 0; bool plain = true;                      // one aligned run, nothing but soft clips around it
                for (uint16_t k = 0; k < n_cig; ++k) {
                    const uint32_t cw = rd32(cig + 4 * k), op = cw & 15u;
                    if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) reflen += cw >> 4;
                    if (op == 0 || op == 7 || op == 8) ++n_run; else if (op != 4) plain = false;
                }
                const int64_t s0 = pos, e0 = (int64_t)pos + reflen;
                const auto iv = tg->touched(refID, s0, e0);
                if (iv.first >= iv.second) continue;
                if (trim && plain && n_run == 1) {
                    // query bases from the first to the last target position of the read (include/smc_b200.h: store_lo / store_len)
                    const int64_t p_lo = std::max(s0, iv.first->first), p_hi = std::min(e0, (iv.second - 1)->second) - 1;
                    const int64_t left_sp = (n_cig > 0 && (rd32(cig) & 15u) == 4) ? (int64_t)(rd32(cig) >> 4) : 0;
                    const int64_t q_lo = (p_lo - s0 + left_sp) & ~1ll, q_hi = p_hi - s0 + left_sp + 1;
                    if (q_lo >= 0 && q_hi <= l_seq && q_hi >= q_lo) { R.store_lo = (uint32_t)q_lo; R.store_len = (uint32_t)(q_hi - q_lo); }
                }
            }
            // identity: BC = parts[-2], readid = ':'.join(parts[:-2])   (smCounter.py:319-325)
            const size_t qn = l_rn ? (size_t)l_rn - 1 : 0;
            long c1 = -1, c2 = -1;                  // last and second-to-last ':'
            for (long k = (long)qn - 1; k >= 0; --k)
                if (qname[k] == ':') { if (c1 < 0) c1 = k; else { c2 = k; break; } }
            if (c1 < 0) { R.bc_off = 0; R.bc_len = 0; R.rid_len = 0; }          // fewer than 2 fields: parts[-2] would raise in Python
            else if (c2 < 0) { R.bc_off = 0; R.bc_len = (uint32_t)c1; R.rid_len = 0; }
            else { R.bc_off = (uint32_t)(c2 + 1); R.bc_len = (uint32_t)(c1 - c2 - 1); R.rid_len = (uint32_t)c2; }
            uint64_t code = 1;
            bool packable = R.bc_len <= 31;
            if (packable)
                for (uint32_t k = 0; k < R.bc_len; ++k) {
                    const char ch = qname[R.bc_off + k];
                    const int v = ch == 'A' ? 0 : ch == 'C' ? 1 : ch == 'G' ? 2 : ch == 'T' ? 3 : -1;
                    if (v < 0) { packable = false; break; }
                    code = (code << 2) | (uint64_t)v;
                }
            R.code = packable ? code : 0;
            uint64_t h1 = 0x243f6a8885a308d3ull ^ R.bc_len, h2 = 0x13198a2e03707344ull + R.rid_len;
            hash_bytes(reinterpret_cast<const uint8_t*>(qname) + R.bc_off, R.bc_len, h1, h2);
            hash_bytes(reinterpret_cast<const uint8_t*>(qname), R.rid_len, h1, h2);
            R.h1 = h1; R.h2 = h2;
            R.keep = 1;
            ++kept_here;
        }
    });
    if (bad_rec.load() != SIZE_MAX) { err = "malformed BAM record (field lengths exceed block_size)"; return -1; }
    n_kept = kept.load();
    if (n_kept >= (1ull << 31)) { err = "more than 2^31 reads"; return -1; }
    return 0;
}

// ---- pass 3a: fragment identities.  first_rec[i] = the first record of kept record i's (barcode, readid) identity.  Threads
// own disjoint hash partitions: each walks the records in order, keeps its identities in its own open-addressing table and
// notes, per record, the FIRST record of that identity (hits verified on the name bytes, so the identities are exact).
static int fragment_firsts(const uint8_t* r, const std::vector<size_t>& offs, const Buf<RecInfo>& info, size_t n, int threads,
                           Buf<uint32_t>& first_rec, std::string& err) {
    const size_t nrec = offs.size();
    if (!first_rec.resize(nrec)) return out_of_memory(err, "the fragment identities");
    auto same_identity = [&](size_t i, size_t j) {
        const RecInfo& A = info[i]; const RecInfo& B = info[j];
        if (A.bc_len != B.bc_len || A.rid_len != B.rid_len) return false;
        const uint8_t* qa = &r[offs[i] + 4 + 32]; const uint8_t* qb = &r[offs[j] + 4 + 32];
        return memcmp(qa + A.bc_off, qb + B.bc_off, A.bc_len) == 0 && memcmp(qa, qb, A.rid_len) == 0;
    };
    const int P = (int)std::max<size_t>(1, std::min<size_t>((size_t)threads, n / 65536 + 1));
    auto part_of = [&](size_t i) { return (int)((info[i].h2 >> 40) % (uint64_t)P); };
    // the kept records of every partition, in record order: counted and filled by ranges of records in parallel, so that a
    // partition's thread walks its own records only (not the whole file once per thread)
    std::vector<uint32_t> plist(n);
    std::vector<size_t> pstart((size_t)P + 1, 0);
    {
        const int T = (int)std::max<size_t>(1, std::min<size_t>((size_t)threads, nrec / 65536 + 1));
        std::vector<size_t> cnt((size_t)T * (size_t)P, 0);
        for_ranges(nrec, T, [&](size_t a, size_t e, int t) {
            std::vector<size_t> c((size_t)P, 0);
            for (size_t i = a; i < e; ++i) if (info[i].keep) ++c[(size_t)part_of(i)];
            for (int q = 0; q < P; ++q) cnt[(size_t)t * P + q] = c[(size_t)q];
        });
        size_t run_tot = 0;
        for (int q = 0; q < P; ++q) {
            pstart[(size_t)q] = run_tot;
            for (int t = 0; t < T; ++t) { const size_t c = cnt[(size_t)t * P + q]; cnt[(size_t)t * P + q] = run_tot; run_tot += c; }
        }
        pstart[(size_t)P] = run_tot;
        for_ranges(nrec, T, [&](size_t a, size_t e, int t) {
            std::vector<size_t> cur((size_t)P);
            for (int q = 0; q < P; ++q) cur[(size_t)q] = cnt[(size_t)t * P + q];
            for (size_t i = a; i < e; ++i) if (info[i].keep) plist[cur[(size_t)part_of(i)]++] = (uint32_t)i;
        });
    }
    for_each_thread(P, [&](int t) {
        struct Ent { uint64_t h1, h2; uint32_t rec; };
        const size_t mine = pstart[(size_t)t + 1] - pstart[(size_t)t];
        size_t cap = 16;
        while (cap < 2 * mine + 2) cap <<= 1;
        std::vector<Ent> tab(cap, Ent{0, 0, UINT32_MAX});
        for (size_t q = pstart[(size_t)t]; q < pstart[(size_t)t + 1]; ++q) {
            const size_t i = plist[q];
            const RecInfo& R = info[i];
            size_t k = (size_t)R.h1 & (cap - 1);
            for (;;) {
                Ent& E = tab[k];
                if (E.rec == UINT32_MAX) { E = Ent{R.h1, R.h2, (uint32_t)i}; first_rec[i] = (uint32_t)i; break; }
                if (E.h1 == R.h1 && E.h2 == R.h2 && same_identity(E.rec, i)) { first_rec[i] = E.rec; break; }
                k = (k + 1) & (cap - 1);
            }
        }
    });
    return 0;
}

// ---- pass 3b: the n output slots and every per-read output array, the payload offsets, the fragment ids (a prefix sum over
// "is a first record" numbers the identities in order of first appearance -- the same ids the sequential dictionary would
// hand out), the barcode dictionary; then the payload arrays, sized by the offsets
static int number_reads(smc_bam* h, const uint8_t* r, const std::vector<size_t>& offs, Buf<RecInfo>& info, const Buf<uint32_t>& first_rec,
                        size_t n, bool trim, int threads, Buf<uint32_t>& slot) {
    const size_t nrec = offs.size();
    Buf<uint32_t> id_of;                                                    // id of the identity whose first record is i
    const bool ok = slot.resize(nrec) && id_of.resize(nrec) && h->ref_id.resize(n) && h->pos.resize(n) && h->nm.resize(n) &&
                    h->l_seq.resize(n) && h->flag.resize(n) && h->n_cigar.resize(n) && h->mapq.resize(n) && h->seq_off.resize(n) &&
                    h->qual_off.resize(n) && h->cigar_off.resize(n) && h->umi.resize(n) && h->frag_id.resize(n) &&
                    h->store_lo.resize(trim ? n : 0) && h->store_len.resize(trim ? n : 0);
    if (!ok) return out_of_memory(h->err, "the read arrays");
    h->dict_umis.clear();
    // exclusive prefix sums over the records (kept reads, identities, payload sizes): per-range totals in parallel, a scan of
    // the few totals, then every range fills its own slice
    struct Tot { size_t o, id, seq, qual, cig; };
    const int T = (int)std::max<size_t>(1, std::min<size_t>((size_t)threads, nrec / 65536 + 1));
    std::vector<Tot> base(T + 1, Tot{0, 0, 0, 0, 0});
    for_ranges(nrec, T, [&](size_t a, size_t e, int t) {
        Tot s{0, 0, 0, 0, 0};
        for (size_t i = a; i < e; ++i) {
            const RecInfo& R = info[i];
            if (!R.keep) continue;
            ++s.o; s.id += first_rec[i] == (uint32_t)i;
            s.seq += ((size_t)R.store_len + 1) / 2; s.qual += (size_t)R.store_len; s.cig += rd16(&r[offs[i] + 4 + 12]);
        }
        base[t + 1] = s;
    });
    for (int t = 0; t < T; ++t) {
        base[t + 1].o += base[t].o; base[t + 1].id += base[t].id; base[t + 1].seq += base[t].seq;
        base[t + 1].qual += base[t].qual; base[t + 1].cig += base[t].cig;
    }
    for_ranges(nrec, T, [&](size_t a, size_t e, int t) {
        Tot s = base[t];
        for (size_t i = a; i < e; ++i) {
            const RecInfo& R = info[i];
            if (!R.keep) continue;
            slot[i] = (uint32_t)s.o;
            h->seq_off[s.o] = (int64_t)s.seq; h->qual_off[s.o] = (int64_t)s.qual; h->cigar_off[s.o] = (int64_t)s.cig;
            if (first_rec[i] == (uint32_t)i) id_of[i] = (uint32_t)s.id++;
            ++s.o; s.seq += ((size_t)R.store_len + 1) / 2; s.qual += (size_t)R.store_len; s.cig += rd16(&r[offs[i] + 4 + 12]);
        }
    });
    // barcodes that do not pack into 64 bits get dictionary codes in order of first appearance (rare: sequential)
    std::unordered_map<std::string, uint64_t> umi_dict;
    std::atomic<int> any_dict(0);
    for_ranges(nrec, T, [&](size_t a, size_t e, int) {
        for (size_t i = a; i < e; ++i) if (info[i].keep && info[i].code == 0) { any_dict = 1; break; }
    });
    for (size_t i = 0; any_dict.load() && i < nrec; ++i) {
        RecInfo& R = info[i];
        if (!R.keep || R.code != 0) continue;
        const std::string bc(reinterpret_cast<const char*>(&r[offs[i] + 4 + 32]) + R.bc_off, R.bc_len);
        auto it = umi_dict.find(bc);
        if (it == umi_dict.end()) {
            R.code = (1ull << 63) | (uint64_t)umi_dict.size();
            umi_dict.emplace(bc, R.code);
            h->dict_umis.push_back(bc);
        } else R.code = it->second;
    }
    for_ranges(nrec, T, [&](size_t a, size_t e, int) {
        for (size_t i = a; i < e; ++i) {
            if (!info[i].keep) continue;
            h->frag_id[slot[i]] = id_of[first_rec[i]];
            h->umi[slot[i]] = info[i].code;
        }
    });
    if (!h->seq.resize(base[T].seq) || !h->qual.resize(base[T].qual) || !h->cigar.resize(base[T].cig)) return out_of_memory(h->err, "the read payloads");
    return 0;
}

// ---- pass 4: scalars and payloads to their slots; the stored qualities are counted on the way (the upload codebook needs to
// know which occur)
static void copy_records(smc_bam* h, const uint8_t* r, const std::vector<size_t>& offs, const Buf<RecInfo>& info, const Buf<uint32_t>& slot,
                         bool trim, int threads) {
    std::vector<std::vector<uint64_t>> qhist((size_t)threads, std::vector<uint64_t>(256, 0));
    parallel_for(offs.size(), threads, [&](size_t a, size_t e, int th) {
        uint32_t hq[4][256];
        memset(hq, 0, sizeof(hq));
        uint64_t since = 0;
        uint64_t* hout = qhist[(size_t)th % qhist.size()].data();
        auto flush = [&]() { for (int c = 0; c < 256; ++c) hout[c] += (uint64_t)hq[0][c] + hq[1][c] + hq[2][c] + hq[3][c]; memset(hq, 0, sizeof(hq)); since = 0; };
        for (size_t i = a; i < e; ++i) {
            if (!info[i].keep) continue;
            const size_t o = slot[i];
            const uint8_t* b = &r[offs[i] + 4];
            const uint8_t* rec_end = b + rdi32(&r[offs[i]]);
            const uint8_t l_rn = b[8];
            const uint16_t n_cig = rd16(b + 12);
            const int32_t l_seq = rdi32(b + 16);
            const uint8_t* cig = b + 32 + l_rn;
            const uint8_t* sq = cig + 4 * (size_t)n_cig;
            const uint8_t* ql = sq + ((size_t)l_seq + 1) / 2;
            h->ref_id[o] = rdi32(b); h->pos[o] = rdi32(b + 4); h->flag[o] = rd16(b + 14); h->mapq[o] = b[9];
            h->nm[o] = first_nm(ql + l_seq, rec_end); h->l_seq[o] = l_seq; h->n_cigar[o] = n_cig;
            const size_t w_lo = info[i].store_lo, w_len = info[i].store_len;
            if (trim) { h->store_lo[o] = (int32_t)w_lo; h->store_len[o] = (int32_t)w_len; }
            if (w_len) memcpy(&h->seq[(size_t)h->seq_off[o]], sq + w_lo / 2, (w_len + 1) / 2);
            if (w_len) memcpy(&h->qual[(size_t)h->qual_off[o]], ql + w_lo, w_len);
            if (n_cig) memcpy(&h->cigar[(size_t)h->cigar_off[o]], cig, 4 * (size_t)n_cig);
            {
                const uint8_t* q = ql + w_lo;
                size_t k = 0;
                for (; k + 4 <= w_len; k += 4) { ++hq[0][q[k]]; ++hq[1][q[k + 1]]; ++hq[2][q[k + 2]]; ++hq[3][q[k + 3]]; }
                for (; k < w_len; ++k) ++hq[0][q[k]];
                since += w_len;
                if (since > (1u << 30)) flush();
            }
        }
        flush();
    });
    for (int c = 0; c < 256; ++c) { h->qual_hist[c] = 0; for (auto& t : qhist) h->qual_hist[c] += t[(size_t)c]; }
}

static void fill_reads(smc_bam* h, size_t n, bool trim, smc_bam_reads* out) {
    out->n_reads = (int64_t)n;
    out->ref_id = h->ref_id.data(); out->pos = h->pos.data(); out->flag = h->flag.data(); out->mapq = h->mapq.data();
    out->nm = h->nm.data(); out->l_seq = h->l_seq.data(); out->seq_off = h->seq_off.data(); out->qual_off = h->qual_off.data();
    out->cigar_off = h->cigar_off.data(); out->n_cigar = h->n_cigar.data(); out->umi = h->umi.data(); out->frag_id = h->frag_id.data();
    out->seq = h->seq.data(); out->seq_bytes = (int64_t)h->seq.size(); out->qual = h->qual.data(); out->qual_bytes = (int64_t)h->qual.size();
    out->cigar = h->cigar.data(); out->n_cigar_words = (int64_t)h->cigar.size(); out->n_dict_umis = (int64_t)h->dict_umis.size();
    out->store_lo = trim ? h->store_lo.data() : nullptr; out->store_len = trim ? h->store_len.data() : nullptr;
    out->qual_hist = h->qual_hist;
}

extern "C" int smc_bam_decode(smc_bam* h, int64_t n_iv, const int32_t* iv_ref, const int32_t* iv_start, const int32_t* iv_end,
                              smc_bam_reads* out) {
    if (!h || !out || (n_iv > 0 && (!iv_ref || !iv_start || !iv_end))) { if (h) h->err = "smc_bam_decode: null argument"; return -2; }
    if (h->decoded) { h->err = "smc_bam_decode: a handle decodes once (the inflated stream is released afterwards); open the file again"; return -2; }
    try {
        const int rc = load_records(h, n_iv, iv_ref, iv_start, iv_end);
        if (rc != 0) { h->decoded = true; return rc; }
        const size_t nref = h->ref_names.size();
        const Targets targets(nref, n_iv, iv_ref, iv_start, iv_end);
        const bool trim = h->trim && n_iv > 0;
        const uint8_t* r = h->raw.data();
        auto pt = phase_timer();
        std::vector<size_t> offs;
        if (record_offsets(r, h->first_record, h->raw.size(), nref, h->threads, offs, h->err) != 0) return -1;
        pt.lap("pass 1 boundaries");
        Buf<RecInfo> info;
        size_t n = 0;
        if (record_fields(r, offs, nref, n_iv > 0 ? &targets : nullptr, trim, h->threads, info, n, h->err) != 0) return -1;
        pt.lap("pass 2 fields + hash");
        Buf<uint32_t> first_rec, slot;
        if (fragment_firsts(r, offs, info, n, h->threads, first_rec, h->err) != 0) return -1;
        pt.lap("fragment identities");
        if (number_reads(h, r, offs, info, first_rec, n, trim, h->threads, slot) != 0) return -1;
        pt.lap("pass 3 numbering + offsets");
        copy_records(h, r, offs, info, slot, trim, h->threads);
        pt.lap("pass 4 copy");
        fill_reads(h, n, trim, out);
    } catch (const std::bad_alloc&) {                 // a std::vector or std::string of the decode did not fit in memory
        return out_of_memory(h->err, "the decode");
    }
    h->raw.resize(0);                              // the inflated stream is not needed any more (one decode per handle)
    h->decoded = true;
    return 0;
}
