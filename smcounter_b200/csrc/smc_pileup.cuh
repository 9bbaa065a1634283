// K1 (read prep / CIGAR walk) and K3 (tile pileup) kernels.
//
// Thread mapping of the pileup kernels ("the transpose"): one warp owns a run of tile events of one tile of 32 consecutive
// target loci, LANE = LOCUS.  The warp streams the tile's reads in (barcode, fragment, BAM index) order; every lane applies
// the read to its own locus.  Barcode and fragment boundaries are therefore warp-uniform, every counter is lane-private
// (no atomics in the loops), and the reference's order-dependent semantics (first read of a fragment defines its base,
// discordant mates delete the fragment, a third read may recreate it -- smCounter.py:467-479) are reproduced by a plain
// per-lane state machine.
//
// K3 is two kernels that meet at a 16-bit "fragment code" per (fragment, locus):
//   k_gather  (K3a)  smCounter.py:368-479   pileup of every read event: base / quality gather, read-level tallies, fragment
//                    merge.  No FP64, few registers, high occupancy: this is where all the DRAM / L2 latency of the path is.
//   k_merge   (K3b)  smCounter.py:26-98, 482-532   per-barcode posterior (calProb), prediction index, consensus counters.
//                    FP64 and 128-bit fixed point; its only input is the coalesced stream of fragment codes.  The rare
//                    barcodes whose calProb takes the general form go to k_merge_deferred, one thread per barcode and locus.
#pragma once
#include "smc_common.cuh"

// ------------------------------------------------------------------------------------------------------------
// K1: per-read preparation: thread r handles read r (inputs coalesced) and writes its records at the read's sorted position.
// Restates smCounter.py:327-356 (mapq, NM, nIndel, leftSP, mismatchPer100b) and the htslib column membership
// pos <= p < reference_end, once per read instead of once per pileup event.
// ------------------------------------------------------------------------------------------------------------

// The 32 bytes of a read the gather loop needs (the 64-byte ReadRec keeps everything, for the rare paths).  Everything that is
// the same for all 32 loci of a tile is resolved here, once per read: the query offset folded into the payload offset, and the
// two "distance to an end" windows of smCounter.py:432-452 as ranges of covered-locus indices.
struct __align__(16) GRec {
    int32_t  lo;         // first covered locus index
    uint32_t gspan_fl;   // bits 0-15: simple reads hi - lo, other reads 0 (the gather loop never covers them); bits 16.. GR_* flags
    uint32_t bq_base;    // quality | BAM nibble << 8 of reference position p is bq[bq_base + p]   (wrapping 32-bit arithmetic)
    uint32_t unused;
    uint32_t le;         // covered loci [lo + (le & 0xffff), lo + (le >> 16)) are within 20 of the barcode end    (:432-452)
    uint32_t ple;        // R2: the same for "within primerDist of the primer end"; empty for R1
    uint32_t urank, frank;
};
static_assert(sizeof(GRec) == 32, "GRec must be 32 bytes");
#define GR_OK      (1u << 16)    // passes the MQ + mismatch gate
#define GR_REVERSE (1u << 17)
#define GR_READ2   (1u << 18)
#define GR_SIMPLE  (1u << 19)

struct PrepArgs {
    int64_t n_reads;
    const uint32_t* inv;          // read index -> srank (sorted position)
    const uint32_t* urank;        // per srank
    const uint32_t* frank;
    const int32_t* ref_id; const int32_t* pos; const uint16_t* flag; const uint8_t* mapq; const int32_t* nm;
    const int32_t* l_seq; const uint32_t* bq_off; const int64_t* cigar_off;   // bq_off: word of the stored window's first base in bq[]
    const int32_t* store_lo; const int32_t* store_len;     // optional stored window of the read's bases / qualities (nullptr: whole read)
    const uint16_t* n_cigar; const uint32_t* cigar;
    const uint64_t* loci_key; int64_t n_loci;
    int minMQ; int primerDist; double mismatchThr;
    ReadRec* recs; GRec* grec; uint32_t* gflags;
    uint8_t* pipe_need; uint32_t pipe_n; const uint32_t* chunk_first;       // pipelined upload only (else pipe_need == nullptr)
};

#define GF_DYN_FULL   1u
#define GF_BAD_READ   2u     // l_seq / clip length beyond the 16-bit record fields
#define GF_CODE_FULL  4u     // a unit ran out of fragment-code storage (host retries with the worst-case layout)
#define GF_BAD_STORE  8u     // stored window (store_lo / store_len) malformed or not covering every target base of the read
#define GF_DEFER_FULL 16u    // k_merge ran out of deferred-barcode records (host retries with a longer list)
#define GF_FRAG_UMI   32u    // a frag_id carries reads of two barcodes (k_umi_slots)

__global__ void __launch_bounds__(256) k_read_prep(PrepArgs A) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;      // BAM order in (coalesced), sorted position out
    if (r >= A.n_reads) return;
    const int64_t s = A.inv[r];
    uint32_t ncig = A.n_cigar[r];
    int64_t co = A.cigar_off[r];
    int32_t lseq = A.l_seq[r];
    int reflen = 0, nindel = 0, leftSP = 0, lead = 0, trail = 0, n_refops = 0;
    bool simple = true, in_lead = true;
    uint32_t c4[4] = {0, 0, 0, 0};
    for (uint32_t k = 0; k < ncig; ++k) {
        uint32_t cw = A.cigar[co + k];
        if (k < 4) c4[k] = cw;
        uint32_t op = cw & 15u; int len = (int)(cw >> 4);
        if (op == 1 || op == 2) nindel += len;                 // smCounter.py:343-344
        if (k == 0 && op == 4) leftSP = len;                   // :345-346
        if (op == 0 || op == 7 || op == 8) { reflen += len; ++n_refops; in_lead = false; trail = 0; }
        else if (op == 2 || op == 3) { reflen += len; simple = false; in_lead = false; trail = 0; }
        else if (op == 4) { if (in_lead) lead += len; else trail += len; }
        else if (op == 5) { simple = false; }
        else { simple = false; in_lead = false; trail = 0; }   // I, P
    }
    if (n_refops != 1) simple = false;
    int alnlen = lseq - lead - trail;                          // query_alignment_length
    int nmv = A.nm[r];
    int mismatch = nmv - nindel; if (mismatch < 0) mismatch = 0;                       // :352
    double mm100 = lseq > 0 ? (100.0 * (double)mismatch) / (double)lseq : 0.0;          // :356
    uint32_t fl = A.flag[r];
    bool ok = ((int)A.mapq[r] >= A.minMQ) && (mm100 <= A.mismatchThr);
    int32_t start = A.pos[r];
    int64_t lo = 0, hi = 0;
    if (!(fl & 0x4u) && reflen > 0) {
        uint64_t k0 = ((uint64_t)(uint32_t)A.ref_id[r] << 32) | (uint32_t)start;
        uint64_t k1 = ((uint64_t)(uint32_t)A.ref_id[r] << 32) | (uint32_t)(start + reflen);
        lo = lower_bound_u64(A.loci_key, A.n_loci, k0);
        hi = lower_bound_u64(A.loci_key, A.n_loci, k1);
    }
    if (lseq > 65535 || leftSP > 65535 || alnlen < 0 || alnlen > 65535) { atomicOr(A.gflags, GF_BAD_READ); lo = hi = 0; }
    ReadRec rec;
    rec.start = start; rec.lo = (int32_t)lo; rec.hi = (int32_t)hi;
    const bool rev = fl & 0x10u, r2 = fl & 0x80u;
    rec.meta = (ok ? RM_OK : 0u) | (rev ? RM_REVERSE : 0u) | (r2 ? RM_READ2 : 0u) | (simple ? RM_SIMPLE : 0u) | (ncig << 8);
    // Stored window: bases [slo, slo + slen) of the read are in bq[] (slo even: the uploaded 4-bit bases start on a byte).  The
    // record keeps the offset of the read's (virtual) base 0, so that every later access is offset + query position in wrapping
    // 32-bit arithmetic.
    const int32_t slo = A.store_lo ? A.store_lo[r] : 0, slen = A.store_len ? A.store_len[r] : lseq;
    if (slo < 0 || (slo & 1) || slen < 0 || slo + slen > lseq || (!simple && (slo != 0 || slen != lseq))) { atomicOr(A.gflags, GF_BAD_STORE); lo = hi = 0; }
    else if (simple && hi > lo) {          // every target base of the read must be stored: query position = p + leftSP - start
        const int32_t q0 = (int32_t)(uint32_t)A.loci_key[lo] + leftSP - start, q1 = (int32_t)(uint32_t)A.loci_key[hi - 1] + leftSP - start;
        if (q0 < slo || q1 >= slo + slen) { atomicOr(A.gflags, GF_BAD_STORE); lo = hi = 0; }
    }
    rec.bq_off = A.bq_off[r] - (uint32_t)slo; rec.unused = 0u;
    rec.cigar_off = (uint32_t)co;
    rec.urank = A.urank[s]; rec.frank = A.frank[s];
    rec.read_idx = r; rec.gspan = simple ? (uint32_t)(hi - lo) : 0u;
    rec.sp_aln = (uint32_t)leftSP | ((uint32_t)alnlen << 16);
    rec.cig[0] = c4[0]; rec.cig[1] = c4[1]; rec.cig[2] = c4[2]; rec.cig[3] = c4[3];
    GRec g;
    g.lo = (int32_t)lo;
    g.gspan_fl = rec.gspan | (ok ? GR_OK : 0u) | (rev ? GR_REVERSE : 0u) | (r2 ? GR_READ2 : 0u) | (simple ? GR_SIMPLE : 0u);
    g.bq_base = rec.bq_off; g.unused = 0u; g.le = 0u; g.ple = 0u;
    g.urank = rec.urank; g.frank = rec.frank;
    if (simple && hi > lo) {
        // One aligned run: the query position of reference position p is p + qk, qk = leftSP - start.
        const int32_t qk = leftSP - start;
        g.bq_base = rec.bq_off + (uint32_t)qk;
        // d = p - start is the distance from the alignment start, alnlen - d from its end.
        //   R1: distToBcEnd = rev ? alnlen - d : d;   R2: distToBcEnd = rev ? d : alnlen - d, distToPrimerEnd = rev ? alnlen - d : d
        // "<= X from the start" is the position window [start, start + X], "<= X from the end" is [start + alnlen - X, inf);
        // as ranges of the covered loci [lo, hi): count of loci below a position (loci of one interval are consecutive positions)
        const int32_t n = (int32_t)(hi - lo);
        const int32_t p_first = (int32_t)(uint32_t)A.loci_key[lo];
        const bool contiguous = (int32_t)(uint32_t)A.loci_key[hi - 1] - p_first == n - 1;
        auto below = [&](int64_t x) -> uint32_t {              // number of covered loci at positions < x
            if (contiguous) { const int64_t c = x - (int64_t)p_first; return (uint32_t)(c < 0 ? 0 : c > n ? n : c); }
            int32_t a0 = 0, b0 = n;
            while (a0 < b0) { const int32_t mid = (a0 + b0) >> 1; if ((int64_t)(int32_t)(uint32_t)A.loci_key[lo + mid] < x) a0 = mid + 1; else b0 = mid; }
            return (uint32_t)a0;
        };
        const bool bc_at_start = (r2 == rev);                 // R1 fwd / R2 rev measure the barcode end from the start
        if (bc_at_start) g.le = below((int64_t)start) | (below((int64_t)start + 21) << 16);
        else g.le = below((int64_t)start + alnlen - 20) | ((uint32_t)n << 16);
        if (r2) {
            if (rev) g.ple = below((int64_t)start + alnlen - A.primerDist) | ((uint32_t)n << 16);
            else if (A.primerDist >= 0) g.ple = below((int64_t)start) | (below((int64_t)start + A.primerDist + 1) << 16);
        }
    }
    {
        const uint4* src = reinterpret_cast<const uint4*>(&rec);
        uint4* dst = reinterpret_cast<uint4*>(&A.recs[s]);
        dst[0] = src[0]; dst[1] = src[1]; dst[2] = src[2]; dst[3] = src[3];
        const uint4* gs = reinterpret_cast<const uint4*>(&g);
        uint4* gd = reinterpret_cast<uint4*>(&A.grec[s]);
        gd[0] = gs[0]; gd[1] = gs[1];
    }
    if (A.pipe_need) {                                         // the chunk this read is expanded with (k_unpack)
        uint32_t c = 0;
        for (uint32_t k = 1; k < A.pipe_n; ++k) if (A.chunk_first[k] <= (uint32_t)r) c = k;
        A.pipe_need[s] = (uint8_t)c;
    }
}

// Per tile event (tile-sorted), derived by k_gather while it stages a batch: bit 0 a new fragment starts here, bit 1 a new
// barcode starts here (both set at the first event of a unit), bit 2 the read is one plain aligned run.
#define EF_FRAG   1u
#define EF_UMI    2u
#define EF_SIMPLE 4u
// Units: a tile's events are cut every `chunk` events, moved forward to the next barcode boundary.  One warp per unit.
__global__ void __launch_bounds__(256)
k_unit_bounds(const uint32_t* __restrict__ tile_off, const uint32_t* __restrict__ unit_off, uint32_t n_tiles, uint32_t chunk,
              const uint32_t* __restrict__ ev_read, const uint32_t* __restrict__ urank, uint32_t* __restrict__ unit_eb,
              uint32_t* __restrict__ unit_ee, uint32_t* __restrict__ unit_tile, uint32_t n_units_cap) {
    const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= n_units_cap) return;
    if (u >= unit_off[n_tiles]) { unit_eb[u] = unit_ee[u] = 0; unit_tile[u] = 0; return; }
    const uint32_t tile = (uint32_t)upper_slot_u32(unit_off, (int64_t)n_tiles + 1, u);
    const uint32_t c = u - unit_off[tile];
    const uint32_t tb = tile_off[tile], te = tile_off[tile + 1];
    auto boundary = [&](uint64_t x64) -> uint32_t {
        if (x64 >= te) return te;
        uint32_t x = (uint32_t)x64;
        while (x < te && urank[ev_read[x]] == urank[ev_read[x - 1]]) ++x;       // x > tb here: forward to the next barcode start
        return x;
    };
    const uint32_t eb = c == 0 ? tb : boundary((uint64_t)tb + (uint64_t)c * chunk);
    const uint32_t ee = boundary((uint64_t)tb + (uint64_t)(c + 1) * chunk);
    unit_eb[u] = eb; unit_ee[u] = ee; unit_tile[u] = tile;
}

// ------------------------------------------------------------------------------------------------------------
// Pipelined upload (smc_call_batch): bases and qualities arrive in up to SMC_PIPE_MAX chunks of equal byte size while the
// read sort / prep / tile sort already run.  k_read_prep records, per read, the chunk its bq[] words are expanded with
// (PrepArgs::pipe_need, k_chunk_need); a unit may start once the latest chunk any of its reads needs is expanded.  Right for
// any payload layout; a payload stored in read order (a BAM decode) makes the units become ready front to back.
// ------------------------------------------------------------------------------------------------------------
#define SMC_PIPE_MAX 16
// first_blocked[c] = smallest unit that has to wait for chunk c + 1 (one warp per unit)
__global__ void __launch_bounds__(256)
k_pipe_unit_need(const uint32_t* __restrict__ unit_eb, const uint32_t* __restrict__ unit_ee, const uint32_t* __restrict__ ev_read,
                 const uint8_t* __restrict__ need, uint32_t n_units, uint32_t* __restrict__ first_blocked) {
    const uint32_t u = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (u >= n_units) return;
    const uint32_t eb = unit_eb[u], ee = unit_ee[u];
    uint32_t m = 0;
    for (uint32_t e = eb + lane; e < ee; e += 32) m = max(m, (uint32_t)__ldg(&need[__ldg(&ev_read[e])]));
    for (int d = 16; d > 0; d >>= 1) m = max(m, __shfl_xor_sync(FULL_MASK, m, d));
    if (lane == 0 && eb < ee && m > 0) atomicMin(&first_blocked[m - 1], u);
}

// ------------------------------------------------------------------------------------------------------------
// Fragment codes: what k_gather hands to k_merge, 16 bits per (fragment, locus); a unit's codes are stored in groups of
// eight per lane (one 128-bit word), so both kernels move them with fully coalesced 512-byte warp transactions.
//   bits 0-7   effective base quality of the fragment (min over a concordant pair)
//   bits 8-10  allele slot A0 C1 DEL2 T3 G4, or 7 = dynamic allele (its row is in the fragment's extension row)
//   bits 11-12 0 no read of the fragment covers the locus; 1 covered (allBcDict, smCounter.py:463-464); 2 covered and a read
//              passed incCond, but no fragment is left (the barcode is a key of bcDict all the same); 3 the fragment is in
//              bcDict when it closes (:467-479)
//   bit  13    ... and it is 'Paired'
//   bit  14    an extension row belongs to this fragment (warp uniform)
//   bit  15    first fragment of a barcode (warp uniform)
// Storage of unit u (events [eb, ee), len = ee - eb): slots [base, base + cap), one slot = 32 lanes x 16 bit;
// codes grow upward in groups of 8 slots, extension rows (32 lanes x u32 = 2 slots: dynamic-allele rows) grow downward.
// With mult = 1 the codes always fit and there is room for (cap - codes) / 2 extension rows; a unit that needs more sets
// GF_CODE_FULL and the host re-runs the batch with mult = 3, which always fits.
// ------------------------------------------------------------------------------------------------------------
#define FC_AID_SH   8u
#define FC_AID_DYN  7u
#define FC_ST_SH    11u
#define FC_PAIRED   (1u << 13)
#define FC_EXT      (1u << 14)
#define FC_UMIFIRST (1u << 15)

__host__ __device__ inline uint64_t unit_slot_base(uint32_t eb, uint32_t u, uint32_t mult) {
    return 8ull * (((uint64_t)mult * eb + 7ull) / 8ull + 3ull * u);
}
__host__ __device__ inline uint32_t unit_slot_cap(uint32_t len, uint32_t mult) {
    return (uint32_t)(8ull * (((uint64_t)mult * len) / 8ull + 2ull));
}
static inline uint64_t code_slots_total(uint64_t ne, uint64_t n_units, uint32_t mult) {
    return 8ull * ((mult * ne + 7ull) / 8ull + 3ull * (n_units + 1ull)) + 16ull;
}

#define NF SMC_NFIXED
#define NDYN 27            // dynamic alleles (indel starts, N / IUPAC bases) of one barcode at one locus: 5 fixed + 27 = the 32
                           // slots of the allele bit mask; a barcode beyond that raises SMC_ST_UMI_OVERFLOW

// The dynamic-allele table, passed BY VALUE to the out-of-line helpers.
struct DynTab {
    unsigned long long* dkey; uint32_t dmask; uint32_t* drep_read; int32_t* drep_qpos; int32_t* dlen;
    int32_t* dcnt; unsigned long long* dlimb; uint8_t* diskey; uint32_t* dcount; uint32_t* gflags;
    const uint16_t* bq; const uint32_t* bq_off;      // bq[] and each read's first stored word (caller's SoA order): long insertions are
                                                     // compared base by base
};

// BAM nibble of A, C, G, T (1, 2, 4, 8) -> field A0 C1 T2 G3 of the packed register counters / allele slot A0 C1 T3 G4
__device__ __forceinline__ uint32_t nib_field(uint32_t nib) { return (0x20310u >> (2u * nib)) & 3u; }
__device__ __forceinline__ bool nib_is_acgt(uint32_t nib) { return (0x0116u >> nib) & 1u; }

// open-addressing table of the non-ACGT/DEL alleles
__device__ __noinline__ uint32_t dyn_lookup(DynTab T, unsigned long long key, uint32_t rep_read, int rep_qpos, int len) {
    uint32_t h = hash64to32(key) & T.dmask;
    for (uint32_t probe = 0; probe <= T.dmask; ++probe) {
        unsigned long long cur = __ldcg(&T.dkey[h]);
        if (cur == key) return h;
        if (cur == DYN_EMPTY) {
            unsigned long long prev = atomicCAS(&T.dkey[h], DYN_EMPTY, key);
            if (prev == DYN_EMPTY) {
                T.drep_read[h] = rep_read; T.drep_qpos[h] = rep_qpos; T.dlen[h] = len;
                uint32_t c = atomicAdd(T.dcount, 1u);
                if (2ull * (c + 1ull) > (unsigned long long)T.dmask + 1ull) atomicOr(T.gflags, GF_DYN_FULL);
                return h;
            }
            if (prev == key) return h;
        }
        h = (h + 1) & T.dmask;
    }
    atomicOr(T.gflags, GF_DYN_FULL);
    return 0;
}

// Insertions longer than 8 bases do not fit the 64-bit key: the key carries a 32-bit hash of the inserted bases and every hit is
// verified by length (dlen) and base by base against the entry's representative read (drep_read / drep_qpos); two different insertions with
// equal hashes chain to separate entries, so alleles are never merged (collision free, like the short ones).
// `my_bq0`: word of this read's query position 0 in bq[]; the representative's comes from bq_off[] (reads with an insertion are
// always stored whole).  drep_read doubles as the "entry published" flag (0xffffffff until the creator is done).
__device__ __noinline__ uint32_t dyn_lookup_long_ins(DynTab T, unsigned long long key, uint32_t rep_read, int rep_qpos, int len, uint32_t my_bq0) {
    uint32_t h = hash64to32(key) & T.dmask;
    for (uint32_t probe = 0; probe <= T.dmask; ++probe) {
        unsigned long long cur = __ldcg(&T.dkey[h]);
        if (cur == DYN_EMPTY) {
            const unsigned long long prev = atomicCAS(&T.dkey[h], DYN_EMPTY, key);
            if (prev == DYN_EMPTY) {
                T.drep_qpos[h] = rep_qpos; T.dlen[h] = len;
                __threadfence();
                atomicExch(&T.drep_read[h], rep_read);
                uint32_t c = atomicAdd(T.dcount, 1u);
                if (2ull * (c + 1ull) > (unsigned long long)T.dmask + 1ull) atomicOr(T.gflags, GF_DYN_FULL);
                return h;
            }
            cur = prev;
        }
        if (cur == key) {
            uint32_t rr;
            while ((rr = *reinterpret_cast<volatile uint32_t*>(&T.drep_read[h])) == 0xffffffffu) { }
            __threadfence();
            const int rq = *reinterpret_cast<volatile int32_t*>(&T.drep_qpos[h]);
            const uint32_t rs0 = T.bq_off[rr];
            // the key carries no length (only the hash seed does): an insertion that is a prefix of the entry's, or the entry's
            // plus more bases, must not match; with equal lengths the comparison also stays inside the representative's insertion
            bool eq = *reinterpret_cast<volatile int32_t*>(&T.dlen[h]) == len;
            for (int t = 1; t <= len && eq; ++t)
                eq = (__ldg(T.bq + (uint32_t)(my_bq0 + (uint32_t)(rep_qpos + t))) >> 8) == (__ldg(T.bq + (uint32_t)(rs0 + (uint32_t)(rq + t))) >> 8);
            if (eq) return h;
        }
        h = (h + 1) & T.dmask;
    }
    atomicOr(T.gflags, GF_DYN_FULL);
    return 0;
}

// ============================================================================================================
// K3a: k_gather
//
// A warp owns one unit (a run of tile events of one 32-locus tile, cut at barcode starts), LANE = LOCUS.  It works in batches
// of up to 32 tile events and always stops a batch at a fragment start, so that a fragment begins and ends in one batch:
//   stage    : lane k loads the GRec of event k and turns everything that is the same for all 32 loci into three 32-bit LANE
//              MASKS (covered / within 20 of the barcode end / within primerDist of the primer end) and a tally class; barcode
//              and fragment boundaries of the batch become warp-uniform bit masks (ranks of neighbouring events, ballots);
//   gather   : KA_GATHER events at a time every lane loads the quality | nibble word of ITS locus (independent loads:
//              ILP + occupancy hide the latency), adds the event to a per-lane CLASS HISTOGRAM in shared memory (one
//              fire-and-forget shared atomic: 16 classes = strand x {lowQ, not included, R1 x le20, R2 x le20 x ple}, the four
//              bases as 8-bit fields of one word) and leaves a 16-bit event code (quality, allele slot, covered / included);
//   fragments: complete fragments of one or two plain aligned reads -- nearly all of them -- get the reference's fragment merge
//              (smCounter.py:467-479) in closed form from their event codes, two fragments per iteration, branch free; anything
//              else (3+ reads, indel / clipped reads, N / IUPAC bases) takes the ordered per-event state machine;
//   emit     : the lane's fragment code goes to a shared-memory staging row; eight rows leave as one 128-bit word per lane.
// Everything rare is out of line: reads with indels / hard clips / several aligned runs (per-event CIGAR walk),
// non-ACGT bases, pairs on a deletion or a dynamic allele.
// ============================================================================================================
#ifndef KA_WARPS
#define KA_WARPS 4
#endif
#ifndef KA_MINBLOCKS
#define KA_MINBLOCKS 7    // B200, cfg2: 4 warps x 6 / 7 / 8 blocks 1.335 / 1.251 / 1.552 ms; 8 warps x 3 / 4 blocks 1.362 / 1.591
#endif
#ifndef KA_GATHER
#define KA_GATHER 4
#endif
// per-warp shared memory (words): event masks 32 x uint4 | payload bases 32 | srank | event codes 32 x 32 x u16 |
// fragment-code staging | class histogram 16 x 32 | (LIST) first-read staging
#define KA_OFF_BASE  128
#define KA_OFF_SRANK (KA_OFF_BASE + 32)
#define KA_OFF_EVC   (KA_OFF_SRANK + 32)
#define KA_OFF_CST   (KA_OFF_EVC + 512)
#define KA_OFF_HIST  (KA_OFF_CST + 128)
#define KA_OFF_FST   (KA_OFF_HIST + 512)
#define KA_WARP_WORDS(LIST) (KA_OFF_FST + ((LIST) ? 256 : 0))
#define KA_LUT_WORDS 36             // the nibble table of k_gather: 17 x uint2, padded to 16 bytes
#define KA_SMEM_BYTES(LIST) (KA_LUT_WORDS * 4 + KA_WARPS * KA_WARP_WORDS(LIST) * 4)

// event code (internal to k_gather).  Staged codes of plain aligned reads: quality in bits 0-7, bits 8-11 the allele slot
// (A0 C1 T3 G4, as in the fragment code) or, with EC_DYN, the BAM nibble of an N / IUPAC base; codes returned by slow_event:
// BAM nibble in bits 8-11
#define SC_AID_SH   8u
#define EC_NIB_SH   8u
#define EC_COVERED  (1u << 12)
#define EC_DYN      (1u << 13)    // regular base that is not A/C/G/T (N / IUPAC): dynamic allele row
#define EC_INC      (1u << 14)    // event passes incCond (:431): it enters bcDict
#define EC_REGULAR  (1u << 15)    // a plain base, not an indel start / in-deletion event
#define EC_LE20     (1u << 16)    // distance to the barcode end <= 20
#define EC_PLE      (1u << 17)    // R2 and distance to the primer end <= primerDist

// tally classes of a regular A/C/G/T event (smCounter.py:423-459): bit 3 reverse strand; low bits 0 low quality, 1 not
// included (MQ / mismatch gate), 2 + le20 included R1, 4 + le20 + 2 ple included R2
#define TC_REVERSE 8u

struct KAArgs {
    const GRec* grec; const ReadRec* recs; const uint32_t* ev_read; const uint32_t* urank_s; const uint32_t* frank_s;
    const uint32_t* unit_eb; const uint32_t* unit_ee; const uint32_t* unit_tile;
    uint32_t unit0, n_units;      // this launch covers units [unit0, n_units)
    uint32_t code_mult;
    const int32_t* loci_pos; int64_t n_loci;
    const uint16_t* bq; const uint32_t* cigar;
    int minBQ, primerDist;
    uint4* codes; uint32_t* unit_nfrag;
    uint32_t* frag_first;         // LIST only: BAM index of the fragment's first passing read, per (slot, lane)
    uint32_t* umi_urank;          // optional (mask / listing): urank of the k-th barcode of unit u at [eb + k]
    int32_t* loc; int32_t* cnt;
    DynTab T;
};

// Tallies of one pileup event whose base is not A/C/G/T (N / IUPAC, smCounter.py:423-457 with that key): rare, so it goes
// straight to the dynamic-allele row with atomics.  Returns the row | (nibble == N) << 31.
__device__ __noinline__ uint32_t dyn_base_event(DynTab T, uint32_t nib, uint32_t locus, uint32_t read_idx, int qpos,
                                                uint32_t flags /* 1 fwd 2 lowq 4 inc 8 r2 16 le20 32 ple */) {
    const uint32_t e = dyn_lookup(T, dyn_make_key(locus, SMC_K_BASE, nib, 0ull), read_idx, qpos, 0);
    int32_t* row = T.dcnt + (size_t)e * SMC_NCNT;
    atomicAdd(&row[SMC_C_ALLELE], 1);
    if (flags & 1u) atomicAdd(&row[SMC_C_FWD], 1);
    if (flags & 2u) atomicAdd(&row[SMC_C_LOWQ], 1);
    if (flags & 4u) {
        if (!(flags & 8u)) { atomicAdd(&row[SMC_C_R1TOT], 1); if (flags & 16u) atomicAdd(&row[SMC_C_R1LE], 1); }
        else {
            atomicAdd(&row[SMC_C_R2TOT], 1);
            if (flags & 16u) atomicAdd(&row[SMC_C_R2LE], 1);
            if (flags & 32u) atomicAdd(&row[SMC_C_R2PLE], 1);
        }
    }
    return e | (nib == 15u ? 0x80000000u : 0u);
}

// Pileup event of a read that is NOT one plain aligned run (indels, hard clips, ...): htslib resolve_cigar2 for the
// lane's position p, then the allele classification of smCounter.py:371-457.  `rw` = the read's ReadRec (global memory).
// Returns {event code, x}:
//   regular base          : EC_REGULAR, nibble in the code (EC_DYN when it is not A/C/G/T; then x = query position)
//   inside a deletion     : x = SMC_A_DEL, bq = minBQ (:416-421)
//   insertion / deletion start (:371-411): x = NF + row; alleleCnt and strand are tallied here
__device__ __noinline__ uint2 slow_event(DynTab T, const uint32_t* __restrict__ rw, const uint32_t* __restrict__ cigar,
                                         const uint16_t* __restrict__ bqp, int32_t p, int32_t Li, int minBQ, int primerDist) {
    const uint32_t meta = __ldg(rw + 3);
    const int32_t start = (int32_t)__ldg(rw + 6), lo = (int32_t)__ldg(rw + 0), hi = (int32_t)__ldg(rw + 7);
    if (!(Li >= lo && Li < hi)) return make_uint2(0u, 0u);
    const bool reverse = meta & RM_REVERSE, read2 = meta & RM_READ2;
    const uint32_t ncig = meta >> 8;
    const uint32_t spa = __ldg(rw + 2);
    const int leftSP = (int)(spa & 0xffffu), alnlen = (int)(spa >> 16);
    const uint32_t bq_off = __ldg(rw + 4), cigar_off = __ldg(rw + 11);
    int qpos = 0, indel = 0; bool isdel = false;
    {
        int x = start, y = 0;
        for (uint32_t k = 0; k < ncig; ++k) {
            const uint32_t cw = __ldg(&cigar[cigar_off + k]);
            const uint32_t op = cw & 15u; const int len = (int)(cw >> 4);
            if (op == 0 || op == 7 || op == 8 || op == 2 || op == 3) {
                if (p < x + len) {                                           // the op that covers p
                    isdel = (op == 2 || op == 3);
                    qpos = isdel ? y : y + (p - x);
                    if (p == x + len - 1 && k + 1 < ncig) {                   // peek the next op
                        const uint32_t c2 = __ldg(&cigar[cigar_off + k + 1]);
                        const uint32_t op2 = c2 & 15u; const int l2 = (int)(c2 >> 4);
                        if (op2 == 2) indel = -l2;
                        else if (op2 == 1) indel = l2;
                        else if (op2 == 6 && k + 2 < ncig) {
                            int l3 = 0;
                            for (uint32_t kk = k + 2; kk < ncig; ++kk) {
                                const uint32_t c3 = __ldg(&cigar[cigar_off + kk]);
                                const uint32_t op3 = c3 & 15u;
                                if (op3 == 1) l3 += (int)(c3 >> 4);
                                else if (op3 == 2 || op3 == 0 || op3 == 3 || op3 == 7 || op3 == 8) break;
                            }
                            if (l3 > 0) indel = l3;
                        }
                    }
                    break;
                }
                x += len;
                if (op == 0 || op == 7 || op == 8) y += len;
            } else if (op == 1 || op == 4) y += len;
        }
    }
    if (indel == 0 && isdel) {                                                 // :416-421
        const bool inc = (meta & RM_OK);                                       // bq = minBQ passes the quality gate
        return make_uint2(((uint32_t)minBQ & 255u) | EC_COVERED | (inc ? EC_INC : 0u), (uint32_t)SMC_A_DEL);
    }
    const uint32_t w = __ldg(bqp + (uint32_t)(bq_off + (uint32_t)qpos));
    const uint32_t nib = w >> 8, bq = w & 255u;
    const bool lowq = (int)bq < minBQ;
    const bool inc = !lowq && (meta & RM_OK);                                  // :378,400,431
    uint32_t code = bq | (nib << EC_NIB_SH) | EC_COVERED | (inc ? EC_INC : 0u);
    if (indel == 0) {                                                          // :423-457 regular base
        const int d = qpos - leftSP;
        const int da = reverse ? alnlen - d : d, db = reverse ? d : alnlen - d;
        if ((read2 ? db : da) <= 20) code |= EC_LE20;
        if (read2 && da <= primerDist) code |= EC_PLE;
        code |= EC_REGULAR;
        if (nib_is_acgt(nib)) return make_uint2(code, 0u);
        return make_uint2(code | EC_DYN, (uint32_t)qpos);
    }
    // insertion start (:371-389) or deletion start (:392-411): alleleCnt and strand only
    unsigned long long key; int len;
    if (indel > 0) {
        len = indel;
        unsigned long long payload;
        if (len <= 8) {
            unsigned long long nibs = 0;
            for (int t = 0; t < len; ++t)
                nibs |= (unsigned long long)(__ldg(bqp + (uint32_t)(bq_off + (uint32_t)(qpos + 1 + t))) >> 8) << (28 - 4 * t);
            payload = ((unsigned long long)len << 32) | nibs;
        } else {
            uint32_t hsh = 2166136261u ^ (uint32_t)len;
            for (int t = 0; t < len; ++t)
                hsh = (hsh ^ (__ldg(bqp + (uint32_t)(bq_off + (uint32_t)(qpos + 1 + t))) >> 8)) * 16777619u;
            payload = (15ull << 32) | hsh;
        }
        key = dyn_make_key((uint32_t)Li, SMC_K_INS, nib, payload);
    } else {
        len = -indel;
        key = dyn_make_key((uint32_t)Li, SMC_K_DEL, nib, (unsigned long long)len);
    }
    const uint32_t e = (indel > 8) ? dyn_lookup_long_ins(T, key, __ldg(rw + 10), qpos, len, bq_off) : dyn_lookup(T, key, __ldg(rw + 10), qpos, len);
    atomicAdd(&T.dcnt[(size_t)e * SMC_NCNT + SMC_C_ALLELE], 1);
    if (!reverse) atomicAdd(&T.dcnt[(size_t)e * SMC_NCNT + SMC_C_FWD], 1);
    return make_uint2(code, NF + e);
}

// concordPairCnt / discordPairCnt of an allele that has no register field ('DEL' or a dynamic allele): rare, atomics
__device__ __noinline__ void pair_bump_global(int32_t* cnt, size_t nl, int64_t L, int32_t* dcnt, uint32_t aid, int which /* SMC_C_CONCORD | SMC_C_DISCORD */) {
    if (aid < NF) atomicAdd(&cnt[((size_t)aid * SMC_NCNT + which) * nl + L], 1);
    else atomicAdd(&dcnt[(size_t)(aid - NF) * SMC_NCNT + which], 1);
}

// state of the lane's open fragment
#define FS_SEEN   1u      // a read of the fragment covers the locus
#define FS_HADINC 2u      // a read passed incCond
#define FS_EXISTS 4u      // the fragment is in bcDict
#define FS_PAIRED 8u

// lanes [a, b) of a warp as a bit mask (a, b any integers)
__device__ __forceinline__ uint32_t lane_range_mask(int a, int b) {
    a = max(a, 0); b = min(b, 32);
    return b > a ? ((0xffffffffu >> (32 - (b - a))) << a) : 0u;
}

// The lane's class histogram (shared memory, word [class][lane], 4 x 8-bit fields A C T G) and its concordant / discordant
// pair counters (registers, same fields) -> the per-locus global accumulators ([field][locus]: coalesced across lanes)
__device__ __forceinline__ void flush_tallies(int32_t* cnt, size_t nl, int64_t L, bool lane_valid, uint32_t* hist_lane, uint32_t& conc, uint32_t& disc) {
    uint32_t h[16];
#pragma unroll
    for (int t = 0; t < 16; ++t) { h[t] = hist_lane[t * 32]; hist_lane[t * 32] = 0u; }
    // no field can overflow: an event adds 1 to one class of one base, and at most 255 events lie between two flushes
    const uint32_t r1le = h[3] + h[11], r1tot = h[2] + h[10] + r1le;
    const uint32_t r2le = h[5] + h[7] + h[13] + h[15], r2ple = h[6] + h[7] + h[14] + h[15];
    const uint32_t r2tot = h[4] + h[5] + h[6] + h[7] + h[12] + h[13] + h[14] + h[15];
    const uint32_t lowq = h[0] + h[8];
    const uint32_t fwd = h[0] + h[1] + h[2] + h[3] + h[4] + h[5] + h[6] + h[7];
    const uint32_t allele = fwd + h[8] + h[9] + h[10] + h[11] + h[12] + h[13] + h[14] + h[15];
    if (lane_valid && (allele | conc | disc)) {
#pragma unroll
        for (int f = 0; f < 4; ++f) {
            const int a = f + (f >> 1);                                     // A0 C1 T3 G4
            int32_t* base = cnt + (size_t)a * SMC_NCNT * nl + L;
            const uint32_t al = (allele >> (8 * f)) & 255u;
            const uint32_t cc = (conc >> (8 * f)) & 255u, dc = (disc >> (8 * f)) & 255u;
            if (al) {
                const uint32_t fw = (fwd >> (8 * f)) & 255u, lq = (lowq >> (8 * f)) & 255u;
                const uint32_t t1 = (r1tot >> (8 * f)) & 255u, l1 = (r1le >> (8 * f)) & 255u;
                const uint32_t t2 = (r2tot >> (8 * f)) & 255u, l2 = (r2le >> (8 * f)) & 255u, pl = (r2ple >> (8 * f)) & 255u;
                atomicAdd(base + (size_t)SMC_C_ALLELE * nl, (int)al);
                if (fw) atomicAdd(base + (size_t)SMC_C_FWD * nl, (int)fw);
                if (al - fw) atomicAdd(base + (size_t)SMC_C_REV * nl, (int)(al - fw));
                if (lq) atomicAdd(base + (size_t)SMC_C_LOWQ * nl, (int)lq);
                if (t1) atomicAdd(base + (size_t)SMC_C_R1TOT * nl, (int)t1);
                if (l1) atomicAdd(base + (size_t)SMC_C_R1LE * nl, (int)l1);
                if (t2) atomicAdd(base + (size_t)SMC_C_R2TOT * nl, (int)t2);
                if (l2) atomicAdd(base + (size_t)SMC_C_R2LE * nl, (int)l2);
                if (pl) atomicAdd(base + (size_t)SMC_C_R2PLE * nl, (int)pl);
            }
            if (cc) atomicAdd(base + (size_t)SMC_C_CONCORD * nl, (int)cc);
            if (dc) atomicAdd(base + (size_t)SMC_C_DISCORD * nl, (int)dc);
        }
    }
    conc = disc = 0u;
}

// register field increment (1 << 8 * field) of allele slot A0 C1 T3 G4
__device__ __forceinline__ uint32_t slot_field_one(uint32_t aid) { return 1u << (((aid * 3u + 1u) << 1) & 0x18u); }

template <bool LIST>
__global__ void __launch_bounds__(KA_WARPS * 32, KA_MINBLOCKS) k_gather_t(const KAArgs A) {
    extern __shared__ __align__(16) uint32_t smem[];
    // BAM nibble -> {register field increment 1 << 8*field (0: not A/C/G/T), event-code bits of a covered base: allele slot << 8,
    // or nibble << 8 | EC_DYN; EC_COVERED}; entry 16 (what the gather reads for a lane the read does not cover): {0, 0}
    uint2* lut = reinterpret_cast<uint2*>(smem);
    if (threadIdx.x <= 16) {
        const uint32_t n = threadIdx.x;
        const uint32_t f = nib_field(n);
        lut[n] = n == 16u ? make_uint2(0u, 0u)
               : nib_is_acgt(n) ? make_uint2(1u << (8u * f), ((f + (f >> 1)) << SC_AID_SH) | EC_COVERED)
                                : make_uint2(0u, (n << EC_NIB_SH) | EC_DYN | EC_COVERED);
    }
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t* ws = smem + KA_LUT_WORDS + (size_t)w * KA_WARP_WORDS(LIST);
    uint4* smask = reinterpret_cast<uint4*>(ws);                      // per event: covered / le20 / ple lane masks, class + flags
    uint32_t* sbase = ws + KA_OFF_BASE;                               // per event: bq_base
    uint32_t* srank_s = ws + KA_OFF_SRANK;
    uint16_t* evc = reinterpret_cast<uint16_t*>(ws + KA_OFF_EVC);     // 32 x 32 event codes of the batch
    uint32_t* cst = ws + KA_OFF_CST;                                  // fragment-code staging: word [k >> 1][lane], half k & 1
    uint32_t* hist_lane = ws + KA_OFF_HIST + lane;                    // class histogram: word [class][lane]
    uint32_t* fst = ws + KA_OFF_FST;                                  // LIST: [k][lane]
#pragma unroll
    for (int t = 0; t < 16; ++t) hist_lane[t * 32] = 0u;
    __syncthreads();

    const uint32_t unit = A.unit0 + blockIdx.x * KA_WARPS + w;
    if (unit >= A.n_units) return;
    const uint32_t eb = A.unit_eb[unit], ee = A.unit_ee[unit];
    if (eb >= ee) { if (lane == 0) A.unit_nfrag[unit] = 0; return; }
    const uint32_t tile = A.unit_tile[unit];
    const uint64_t so = unit_slot_base(eb, unit, A.code_mult);
    const uint32_t cap = unit_slot_cap(ee - eb, A.code_mult);

    const int64_t L = (int64_t)tile * 32 + lane;
    const bool lane_valid = L < A.n_loci;
    const uint32_t validmask = __ballot_sync(FULL_MASK, lane_valid);
    const int32_t p = lane_valid ? A.loci_pos[L] : 0;
    const int32_t Li = lane_valid ? (int32_t)L : -1;                  // -1 is never inside a read's [lo, hi)
    const uint32_t lanebit = 1u << lane;
    const int32_t tile0 = (int32_t)(tile * 32u);
    const size_t nl = (size_t)A.n_loci;
    const int minBQ = A.minBQ;
    const uint16_t* __restrict__ bqp = A.bq;

    uint32_t conc = 0, disc = 0;                                      // 4 x 8-bit fields (A, C, T, G)
    int cvg = 0;
    // open fragment of this lane: FS_* bits, allele (slot, or NF + dynamic row), effective quality
    uint32_t fs = 0, f_mid = 0, f_bq = 0, f_first = 0xffffffffu;
    // warp-uniform
    uint32_t fcount = 0, ext = 0, umi_k = 0, since_flush = 0;
    uint32_t carry_ur = 0xffffffffu, carry_fr = 0xffffffffu;          // ranks of the previous batch's last event
    bool open = false, umi_first = true, dead = false;
    uint32_t simplemask_cur = 0;                                      // "plain aligned run" bits of the staged batch
    uint16_t* const cst16 = reinterpret_cast<uint16_t*>(cst) + 2 * lane;

    auto flush_codes = [&](uint32_t f0) {
        if (f0 + 8u + 2u * ext > cap) { if (!dead && lane == 0) atomicOr(A.T.gflags, GF_CODE_FULL); dead = true; }
        if (dead) return;
        const uint4 v = make_uint4(cst[lane], cst[32 + lane], cst[64 + lane], cst[96 + lane]);
        A.codes[((so + f0) >> 3) * 32 + lane] = v;
        if (LIST) {
#pragma unroll
            for (int k = 0; k < 8; ++k) A.frag_first[(so + f0 + k) * 32 + lane] = fst[k * 32 + lane];
        }
    };
    // a finished fragment code goes to the staging rows; eight rows are written out as one 128-bit word per lane
    auto put_code = [&](uint32_t code) {
        const uint32_t k = fcount & 7u;
        cst16[((k >> 1) << 6) + (k & 1u)] = (uint16_t)code;
        ++fcount;
        if ((fcount & 7u) == 0u) flush_codes(fcount - 8u);
    };
    // close the open fragment of the ordered pass
    auto emit = [&]() {
        const bool dynl = (fs & FS_EXISTS) && f_mid >= NF;
        const bool any_dyn = __any_sync(FULL_MASK, dynl);
        const uint32_t st = (fs & FS_EXISTS) ? 3u : ((fs & 3u) - ((fs >> 1) & 1u));
        const uint32_t code = (st << FC_ST_SH) | ((fs & FS_PAIRED) ? FC_PAIRED : 0u) | (any_dyn ? FC_EXT : 0u) | (umi_first ? FC_UMIFIRST : 0u) |
                              ((f_mid < NF ? f_mid : FC_AID_DYN) << FC_AID_SH) | f_bq;
        if (LIST) fst[(fcount & 7u) * 32 + lane] = f_first;
        if (any_dyn) {                                                   // extension row: the dynamic-allele rows of this fragment
            if (8u * ((fcount >> 3) + 1u) + 2u * (ext + 1u) > cap) { if (!dead && lane == 0) atomicOr(A.T.gflags, GF_CODE_FULL); dead = true; }
            if (!dead) reinterpret_cast<uint32_t*>(A.codes)[(so + cap - 2u * (ext + 1u)) * 16 + lane] = dynl ? f_mid - NF : 0u;
            ++ext;
        }
        put_code(code);
        fs = 0; f_first = 0xffffffffu; umi_first = false;
    };
    // warp-uniform bookkeeping at the first fragment of a barcode
    auto umi_begin = [&](int j) {
        if (A.umi_urank) { if (lane == 0) A.umi_urank[eb + umi_k] = __ldg(&A.urank_s[srank_s[j]]); ++umi_k; }
    };
    // fragment merge of an event that passed incCond (smCounter.py:467-479); `one` = register field of an A/C/G/T base, else 0
    auto merge = [&](uint32_t mid, uint32_t bq, bool isN, uint32_t one, int j) {
        if (LIST) f_first = min(f_first, __ldg(&A.recs[srank_s[j]].read_idx));
        if (!(fs & FS_EXISTS)) { fs = (fs | FS_HADINC | FS_EXISTS) & ~FS_PAIRED; f_mid = mid; f_bq = bq; }
        else if (mid == f_mid || isN) {
            f_bq = min(f_bq, bq); fs |= FS_PAIRED;
            if (mid == f_mid) {
                if (one) conc += one;
                else pair_bump_global(A.cnt, nl, L, A.T.dcnt, mid, SMC_C_CONCORD);
            }
        } else {
            fs &= ~FS_EXISTS;
            if (one) disc += one;
            else pair_bump_global(A.cnt, nl, L, A.T.dcnt, mid, SMC_C_DISCORD);
        }
    };
    // one pileup event of the ordered pass: the staged event code of a plain aligned read, or the per-event CIGAR walk of any
    // other read (out of line); then the fragment merge
    auto gen_event = [&](int e) {
        uint32_t cd, mid, one; bool isN = false;
        if ((simplemask_cur >> e) & 1u) {
            cd = evc[e * 32 + lane];
            mid = (cd >> SC_AID_SH) & 15u;
            one = slot_field_one(mid);
            if (cd & EC_DYN) {                                                   // rare: N / IUPAC base -> dynamic allele row
                const uint4 m = smask[e];
                const uint32_t* rw = reinterpret_cast<const uint32_t*>(&A.recs[srank_s[e]]);
                const int qpos = p - (int32_t)__ldg(rw + 6) + (int)(__ldg(rw + 2) & 0xffffu);       // p - start + leftSP
                const uint32_t dfl = ((m.w & TC_REVERSE) ? 0u : 1u) | ((int)(cd & 255u) < minBQ ? 2u : 0u) | ((cd & EC_INC) ? 4u : 0u) |
                                     ((m.w & 4u) ? 8u : 0u) | ((m.y & lanebit) ? 16u : 0u) | ((m.z & lanebit) ? 32u : 0u);
                const uint32_t en = dyn_base_event(A.T, mid, (uint32_t)Li, __ldg(rw + 10), qpos, dfl);
                mid = NF + (en & 0x7fffffffu); isN = en >> 31; one = 0;
            }
        } else {                                                             // rare: per-event CIGAR walk, out of line
            const uint32_t* rw = reinterpret_cast<const uint32_t*>(&A.recs[srank_s[e]]);
            const uint2 ev = slow_event(A.T, rw, A.cigar, bqp, p, Li, minBQ, A.primerDist);
            cd = ev.x; mid = ev.y; one = 0;
            if (cd & EC_COVERED) {
                const uint32_t meta = __ldg(rw + 3);
                const bool lowq = (int)(cd & 255u) < minBQ;
                cvg++;
                if (cd & EC_REGULAR) {
                    if (!(cd & EC_DYN)) {
                        const uint2 lv = lut[(cd >> EC_NIB_SH) & 15u];
                        one = lv.x; mid = (lv.y >> SC_AID_SH) & 15u;
                        const uint32_t cls = ((meta & RM_REVERSE) ? TC_REVERSE : 0u) |
                                             (lowq ? 0u : !(cd & EC_INC) ? 1u : (meta & RM_READ2) ? 4u + ((cd & EC_LE20) ? 1u : 0u) + ((cd & EC_PLE) ? 2u : 0u)
                                                                                                   : 2u + ((cd & EC_LE20) ? 1u : 0u));
                        atomicAdd(&hist_lane[cls * 32], one);
                    } else {
                        const uint32_t dfl = ((meta & RM_REVERSE) ? 0u : 1u) | (lowq ? 2u : 0u) | ((cd & EC_INC) ? 4u : 0u) |
                                             ((meta & RM_READ2) ? 8u : 0u) | ((cd & EC_LE20) ? 16u : 0u) | ((cd & EC_PLE) ? 32u : 0u);
                        const uint32_t en = dyn_base_event(A.T, (cd >> EC_NIB_SH) & 15u, (uint32_t)Li, __ldg(rw + 10), (int)ev.y, dfl);
                        mid = NF + (en & 0x7fffffffu); isN = en >> 31;
                    }
                } else if (mid == (uint32_t)SMC_A_DEL) {
                    atomicAdd(&A.cnt[((size_t)SMC_A_DEL * SMC_NCNT + SMC_C_ALLELE) * nl + L], 1);   // alleleCnt only (:416-421, :459)
                }
            }
        }
        if (cd & EC_COVERED) fs |= FS_SEEN;                                  // :463-464
        if (cd & EC_INC) merge(mid, cd & 255u, isN, one, e);                 // :467-479
    };

    for (uint32_t base = eb; base < ee;) {
        const int nb = (int)min(32u, ee - base);
        // ---------------- stage: lane k owns event k
        // boundaries from the dense barcode / fragment ranks of consecutive events (a unit always starts at a barcode start);
        // slots past the end: an empty simple read, no boundary
        uint4 g0 = make_uint4(0u, GR_SIMPLE, 0u, 0u), g1 = make_uint4(0u, 0u, 0xffffffffu, 0xffffffffu);
        uint32_t sr = 0;
        if (lane < nb) {
            sr = __ldg(&A.ev_read[base + lane]);
            const uint4* src = reinterpret_cast<const uint4*>(&A.grec[sr]);
            g0 = __ldg(src); g1 = __ldg(src + 1);                            // lo gspan|flags bq_base unused | le ple urank frank
        }
        uint32_t pur = __shfl_up_sync(FULL_MASK, g1.z, 1), pfr = __shfl_up_sync(FULL_MASK, g1.w, 1);
        if (lane == 0) { pur = carry_ur; pfr = carry_fr; }
        const bool ub = lane < nb && g1.z != pur;
        const bool fb = lane < nb && (ub || g1.w != pfr);
        const uint32_t fragmask = __ballot_sync(FULL_MASK, fb);
        const uint32_t umimask = __ballot_sync(FULL_MASK, ub);
        const uint32_t simplemask = __ballot_sync(FULL_MASK, (g0.y & GR_SIMPLE) != 0u);
        simplemask_cur = simplemask;
        // Events consumed from this batch: when more events follow, stop before the last fragment start, so that a fragment
        // that starts in a batch also ends in it (a fragment of 32+ events is carried across batches by the ordered pass).
        int ncons = nb;
        bool tail_open = false;
        if (base + (uint32_t)nb < ee) {
            const int last = 31 - __clz((int)(fragmask | 1u));
            if (last > 0) ncons = last; else tail_open = true;
        }
        carry_ur = __shfl_sync(FULL_MASK, g1.z, ncons - 1); carry_fr = __shfl_sync(FULL_MASK, g1.w, ncons - 1);
        {
            // what is the same for all 32 loci, as lane masks: covered loci [lo, lo + gspan), the two end-distance windows
            // (only ever needed for included reads); tally class of the read
            const int rel = (int32_t)g0.x - tile0;
            const bool live = lane < ncons;
            const uint32_t okm = (g0.y & GR_OK) ? 0xffffffffu : 0u;
            const uint32_t cov = live ? lane_range_mask(rel, rel + (int)(g0.y & 0xffffu)) & validmask : 0u;
            const uint32_t le = cov & okm & lane_range_mask(rel + (int)(g1.x & 0xffffu), rel + (int)(g1.x >> 16));
            const uint32_t ple = cov & okm & lane_range_mask(rel + (int)(g1.y & 0xffffu), rel + (int)(g1.y >> 16));
            const uint32_t cls = ((g0.y & GR_REVERSE) ? TC_REVERSE : 0u) | (!(g0.y & GR_OK) ? 1u : (g0.y & GR_READ2) ? 4u : 2u);
            smask[lane] = make_uint4(cov, le, ple, cls | ((g0.y & GR_OK) ? EC_INC : 0u));
            sbase[lane] = g0.z;
            srank_s[lane] = sr;
        }
        if (since_flush + 32u > 255u) { flush_tallies(A.cnt, nl, L, lane_valid, hist_lane, conc, disc); since_flush = 0; }
        since_flush += (uint32_t)ncons;
        __syncwarp();
        // ---------------- gather + tally (order independent) of the plain aligned reads, KA_GATHER events at a time
#pragma unroll 1
        for (int g = 0; g < ncons; g += KA_GATHER) {
            uint32_t wv[KA_GATHER];
            uint4 mk[KA_GATHER];
#pragma unroll
            for (int u = 0; u < KA_GATHER; ++u) {
                mk[u] = smask[g + u];
                wv[u] = (mk[u].x & lanebit) ? __ldg(bqp + (sbase[g + u] + (uint32_t)p)) : 16u << 8;    // not covered: lut[16]
            }
#pragma unroll
            for (int u = 0; u < KA_GATHER; ++u) {
                const uint32_t fw = mk[u].w;
                const bool cov = mk[u].x & lanebit;
                const uint32_t bq = wv[u] & 255u;                                    // 0 when not covered
                const uint2 lv = lut[wv[u] >> 8];
                const uint32_t one = lv.x;                                           // 0 when not covered or not A/C/G/T
                const bool lowq = (int)bq < minBQ;
                const uint32_t inc = (cov && !lowq) ? (fw & EC_INC) : 0u;           // :431
                cvg += cov ? 1 : 0;                                                  // :368
                uint32_t cls = fw & 15u;                                             // :428-459, as one class count
                if (mk[u].y & lanebit) cls += 1u;
                if (mk[u].z & lanebit) cls += 2u;
                if (lowq) cls = fw & TC_REVERSE;
                atomicAdd(&hist_lane[cls * 32], one);                                // fire and forget; adds 0 for a lane the read does not cover
                evc[(g + u) * 32 + lane] = (uint16_t)(bq | lv.y | inc);
            }
        }
        // fragment structure of the batch, one event per lane: which fragments are complete runs of one or two plain
        // aligned reads (fast path), and which of those have two reads
        uint32_t fastmask, twomask;
        {
            const uint32_t restk = __funnelshift_rc(fragmask, 0u, (uint32_t)lane + 1u);      // fragmask >> (lane + 1)
            int endk = restk ? lane + __ffs((int)restk) : 32;
            endk = min(endk, ncons);
            const int nk = endk - lane;
            const uint32_t m2 = nk == 2 ? 3u : 1u;
            const bool fastk = !LIST && lane < ncons && ((fragmask >> lane) & 1u) && (endk < ncons || !tail_open) && nk <= 2 &&
                               ((simplemask >> lane) & m2) == m2;
            fastmask = __ballot_sync(FULL_MASK, fastk);
            twomask = __ballot_sync(FULL_MASK, fastk && nk == 2);
        }
        int j = 0;
#pragma unroll 1
        while (j < ncons) {
            if ((fastmask >> j) & 1u) {
                // ---------------- fast path: complete fragments of one or two plain aligned reads, two fragments at a time:
                // the fragment merge of (at most) two reads in BAM order (smCounter.py:467-479) in closed form
                const int n = 1 + (int)((twomask >> j) & 1u);
                const int j2 = j + n;
                const int n2 = (__funnelshift_rc(fastmask, 0u, (uint32_t)j2) & 1u) ? 1 + (int)(__funnelshift_rc(twomask, 0u, (uint32_t)j2) & 1u) : 0;
                const uint16_t* ev = evc + lane;
                uint32_t c[4];
                c[0] = ev[j * 32];
                c[1] = n == 2 ? ev[(j + 1) * 32] : 0u;
                c[2] = n2 ? ev[j2 * 32] : 0u;
                c[3] = n2 == 2 ? ev[(j2 + 1) * 32] : 0u;
                if (!__any_sync(FULL_MASK, ((c[0] | c[1] | c[2] | c[3]) & EC_DYN) != 0u)) {
                    if (open) { emit(); open = false; }                                 // a carried fragment ends here
                    uint32_t codes2[2];
#pragma unroll
                    for (int f = 0; f < 2; ++f) {
                        const uint32_t c0 = c[2 * f], c1 = c[2 * f + 1];
                        const uint32_t i0 = (c0 >> 14) & 1u, i1 = (c1 >> 14) & 1u;        // included
                        const uint32_t both = i0 & i1;
                        const uint32_t same = ((c0 ^ c1) & (15u << SC_AID_SH)) == 0u ? 1u : 0u;
                        const uint32_t one1 = slot_field_one((c1 >> SC_AID_SH) & 15u);
                        conc += (both & same) ? one1 : 0u;                              // keyed by the later read's base
                        disc += (both & (same ^ 1u)) ? one1 : 0u;
                        const uint32_t sel = i0 ? c0 : c1;
                        const uint32_t bqf = both ? min(c0 & 255u, c1 & 255u) : (sel & 255u);
                        const uint32_t exists = both ? same : (i0 | i1);
                        const uint32_t st = exists ? 3u : (i0 | i1) ? 2u : (((c0 | c1) >> 12) & 1u);
                        codes2[f] = (st << FC_ST_SH) | ((both & same) << 13) | (sel & (7u << FC_AID_SH)) | bqf;
                    }
                    const bool us1 = (umimask >> j) & 1u;
                    if (us1) umi_begin(j);
                    put_code(codes2[0] | (us1 ? FC_UMIFIRST : 0u));
                    if (n2) {
                        const bool us2 = (umimask >> j2) & 1u;
                        if (us2) umi_begin(j2);
                        put_code(codes2[1] | (us2 ? FC_UMIFIRST : 0u));
                    }
                    j = j2 + n2;
                    continue;
                }
                // a lane sees an N / IUPAC base in one of these reads: fragment A takes the ordered pass below
            }
            // ---------------- ordered pass over the segment: fragment boundary, per-event merge, the rare events
            const uint32_t rest = __funnelshift_rc(fragmask, 0u, (uint32_t)j + 1u);
            int n = rest ? __ffs((int)rest) : 32;                              // the segment that starts at event j: up to the next fragment start
            n = min(n, ncons - j);
            if ((fragmask >> j) & 1u) {
                if (open) emit();
                umi_first = (umimask >> j) & 1u;
                if (umi_first) umi_begin(j);
                open = true;
            }
#pragma unroll 1
            for (int e = j; e < j + n; ++e) gen_event(e);
            if ((j + n < ncons) || !tail_open) { emit(); open = false; }        // the fragment is complete
            j += n;
        }
        __syncwarp();
        base += (uint32_t)ncons;
    }
    // ---- close a fragment that is still open, write the partial group, flush the tallies
    if (open) emit();
    if (fcount & 7u) flush_codes(fcount & ~7u);
    if (lane == 0) A.unit_nfrag[unit] = dead ? 0u : fcount;
    flush_tallies(A.cnt, nl, L, lane_valid, hist_lane, conc, disc);
    if (lane_valid && cvg) atomicAdd(&A.loc[(size_t)SMC_L_CVG * nl + L], cvg);
}

// ============================================================================================================
// K3b: k_merge -- per-barcode posterior, prediction index, consensus (smCounter.py:26-98, 482-532)
// ============================================================================================================
#ifndef KB_WARPS
#define KB_WARPS 4
#endif
#ifndef KB_MINBLOCKS
#define KB_MINBLOCKS 7    // B200, cfg2: 5 / 6 / 7 / 8 blocks of 4 warps 1.070 / 0.984 / 0.954 / 0.961 ms; 8 warps x 3 / 4 blocks 1.003 / 0.974
#endif
#define KB_FC_WORDS    (NF * 32)                // MTCnt | strongMTCnt << 16 per fixed allele and lane
#define KB_LIMB_WORDS  (NF * 4 * 32)            // 128-bit fixed-point PI accumulator per fixed allele and lane
#define KB_WARP_WORDS  (KB_FC_WORDS + KB_LIMB_WORDS)
#define KB_TAB_BYTES   2064                     // 1 - p of a fragment: entry 0 = not 'Paired' (p = 0.1), entry 1 + quality = 'Paired' (257 doubles, padded to 16 B)
#define KB_SMEM_BYTES  (KB_TAB_BYTES + KB_WARPS * KB_WARP_WORDS * 4)
#define KD_THREADS     128                      // k_merge_deferred

// A barcode whose calProb takes the general form (several alleles, a DEL or dynamic allele, or more fragments than the prior
// table holds) is left by k_merge to k_merge_deferred, in a record of the list KBArgs::defer:
//   {unit, the barcode's first fragment code in the unit, extension rows of the unit before that code, lane | DR_* bits}.
// Such pairs are rare (cfg2: one per ~400 tile events); k_merge keeps neither their per-allele products nor their dynamic-allele
// slots, which keeps its registers and shared memory to what the single-allele barcodes need.
#define DR_STATUS_ONLY (1u << 8)     // a barcode outside the call (masked out, or n <= mtDrop): replayed only for SMC_ST_UMI_OVERFLOW

struct KBArgs {
    const uint4* codes; const uint32_t* unit_nfrag; const uint32_t* frag_first; const uint32_t* umi_urank;
    const uint32_t* unit_eb; const uint32_t* unit_ee; const uint32_t* unit_tile;
    uint32_t unit0, n_units;      // this launch covers units [unit0, n_units)
    uint32_t code_mult;
    int64_t n_loci;
    const double* bqtab;            // [256]  10^(-bq/10), host glibc pow (smCounter.py:469)
    const double* pcrtab;           // [3][(nmax+1)(nmax+2)/2]  10^(-6 (cnt+.5)/(n+.5k)), k = 4,5,6 (smCounter.py:80-81)
    int pcr_nmax; int mtDrop; double smt;
    const int32_t* keep_idx; const int64_t* keep_off; const uint64_t* keep_umi; const uint64_t* umi_of_urank;
    int32_t* loc; int32_t* cnt; unsigned long long* limb;
    DynTab T;
    // optional: list the barcodes of bcDict for flagged loci (down-sampling support)
    const int32_t* list_idx; uint32_t* list_count; const int64_t* list_off; uint64_t* list_umi; uint32_t* list_first; int64_t list_cap;
    uint4* defer; uint32_t defer_cap; uint32_t* defer_count;      // deferred barcodes (GF_DEFER_FULL when the list is full)
};

// A non-negative double < 2^20 as a 128-bit fixed-point integer with LSB 2^-PI_FIX_LSB (= 2^-80), truncated: the integer part
// of l * 2^16 is the high word, the fraction * 2^64 the low word.  Both scalings and the subtraction are exact; the
// truncation drops < 2^-80 per term and is the same whatever the order of the terms, so the sums stay order independent.
__device__ __forceinline__ void pi_fixed128(double l, unsigned long long& lo, unsigned long long& hi) {
    static_assert(PI_FIX_LSB == 80, "pi_fixed128 assumes LSB 2^-80");
    const double t = l * 65536.0;
    hi = __double2ull_rz(t);
    const double frac = t - __ull2double_rz(hi);
    lo = __double2ull_rz(frac * 18446744073709551616.0);
}
__device__ __forceinline__ void add128(unsigned long long& lo, unsigned long long& hi, unsigned long long alo, unsigned long long ahi) {
    lo += alo; hi += ahi + (lo < alo ? 1ull : 0ull);
}
__device__ __forceinline__ void sub128(unsigned long long& lo, unsigned long long& hi, unsigned long long blo, unsigned long long bhi) {
    const unsigned long long borrow = lo < blo ? 1ull : 0ull;
    lo -= blo; hi -= bhi + borrow;
}
// 128-bit value -> three 44-bit carry-save limbs of the global accumulators (v = l0 + l1*2^44 + l2*2^88)
__device__ __forceinline__ void split_limbs(unsigned long long lo, unsigned long long hi, unsigned long long& a0, unsigned long long& a1,
                                            unsigned long long& a2) {
    const unsigned long long M44 = (1ull << 44) - 1ull;
    a0 = lo & M44;
    a1 = ((lo >> 44) | (hi << 20)) & M44;
    a2 = hi >> 24;
}
// a 128-bit PI term or sum -> adds its limbs to the global accumulator l[0], l[stride], l[2 * stride]
__device__ __forceinline__ void add_limbs(unsigned long long* l, size_t stride, unsigned long long lo, unsigned long long hi) {
    unsigned long long a0, a1, a2;
    split_limbs(lo, hi, a0, a1, a2);
    if (a0) atomicAdd(l, a0);
    if (a1) atomicAdd(l + stride, a1);
    if (a2) atomicAdd(l + 2 * stride, a2);
}

// per-lane flags of the open barcode
#define LF_UMI_SEEN  (1u << 0)    // a read of the barcode covers the locus
#define LF_UMI_BC    (1u << 1)    // the barcode is in bcDict (a read passed incCond)
#define LF_DEFER     (1u << 2)    // a fragment showed a second allele or a dynamic one: k_merge_deferred finishes the barcode

struct MergeState {
    // locus-level
    int allFrag, allMT, usedFrag, nBC, usedMT, mt3, mt5, mt7, mt10;
    uint32_t keymask;
    unsigned long long pad_lo, pad_hi;      // PI terms that go to all of A, C, G, T (single-allele barcodes, see umi_finalize)
    uint32_t flags;                         // LF_*
    // barcode-level: until LF_DEFER the barcode has shown one allele, so its product over fragments is rightP and its count n
    int n; uint32_t exist; double rightP; uint32_t last_aid;
    uint32_t first_read;                    // BAM index of the barcode's first passing read at this locus (listing only)
};

#define FCW(a)      fc[(a) * 32 + lane]
#define LIMB(a)     limb[(a) * 32 + lane]

// MTCnt / strongMTCnt of an allele that may be dynamic; add = 1 (MTCnt) or 0x10001 (both)
__device__ __forceinline__ void bump_mt(int32_t* dcnt, int* fc, int lane, uint32_t aid, uint32_t add) {
    if (aid < NF) FCW(aid) += (int)add;
    else {
        int32_t* row = dcnt + (size_t)(aid - NF) * SMC_NCNT;
        atomicAdd(&row[SMC_C_MT], 1);
        if (add >> 16) atomicAdd(&row[SMC_C_STRONG], 1);
    }
}

// A deferred barcode at one locus, as k_merge_deferred rebuilds it (one thread, local memory): allele slots 0 .. NF - 1 are
// the fixed alleles, slot NF + k the barcode's k-th dynamic allele (its row of the dynamic-allele table is dyn[k]).
struct UmiState {
    int n; uint32_t exist; double Q, rightP; uint32_t last_aid; int ndyn; uint32_t status;
    int cnt[NF + NDYN]; double prod[NF + NDYN]; uint32_t dyn[NDYN];
};

// While a barcode shows one allele, its count is n and its product over fragments rightP; its slot is filled when a second
// allele joins, or before umi_general.
__device__ __forceinline__ void umi_fill_single(UmiState& U) {
    const int s0 = __ffs(U.exist) - 1;
    U.cnt[s0] = U.n; U.prod[s0] = U.rightP;
}

// one fragment of bcDict joins the barcode (the per-fragment part of calProb, smCounter.py:56-77)
__device__ __forceinline__ void fragment_join(double p, double q1, uint32_t aid, UmiState& U) {
    int slot = (int)aid;
    if (aid >= NF) {
        const uint32_t e = aid - NF;
        int k = 0;
        while (k < U.ndyn && U.dyn[k] != e) ++k;
        if (k == U.ndyn) {
            if (k < NDYN) { U.dyn[k] = e; U.ndyn = k + 1; }
            else { U.status |= SMC_ST_UMI_OVERFLOW; k = 0; }
        }
        slot = NF + k;
    }
    const uint32_t bit = 1u << slot;
    if (U.exist == 0) U.exist = bit;
    else {
        const bool multi = (U.exist & (U.exist - 1u)) != 0u;
        if (multi || U.exist != bit) {
            if (!multi) umi_fill_single(U);
            if (!(U.exist & bit)) { U.exist |= bit; U.cnt[slot] = 0; U.prod[slot] = U.Q; }
            uint32_t m = U.exist;
            while (m) {                                                  // :70-74
                int s = __ffs(m) - 1; m &= m - 1;
                U.prod[s] = __dmul_rn(U.prod[s], s == slot ? q1 : p);
            }
            U.cnt[slot] += 1;
        }
    }
    U.Q = __dmul_rn(U.Q, p);
    U.rightP = __dmul_rn(U.rightP, q1);                              // :77
    U.n += 1;
    U.last_aid = aid;
}

// PCR prior outside the host-built table (barcodes with > pcr_nmax fragments or > 6 distinct alleles): device pow()
__device__ __noinline__ double pcr_slow(int cnt, double denom) {
    return pow(10.0, -6.0 * (((double)cnt + 0.5) / denom));
}

// -log10(x) for a normal x > 0: x = 2^e m with m in [sqrt(1/2), sqrt(2)), log(m) = 2 atanh(s), s = (m - 1) / (m + 1),
// |s| <= 0.1716; the series is cut after s^21 / 21 (next term < 3e-17 relative).  Within ~2 ulp of the correctly rounded
// value, i.e. ~4e-16 relative on a prediction index that has to match to 1e-9 -- at half the instructions of log10().
__device__ __forceinline__ double neg_log10_normal(double x) {
    const long long b = __double_as_longlong(x);
    int e = (int)(b >> 52) - 1023;
    double m = __longlong_as_double((b & 0x000fffffffffffffll) | 0x3ff0000000000000ll);
    if (m > 1.4142135623730951) { m *= 0.5; e += 1; }
    const double s = (m - 1.0) / (m + 1.0);
    const double z = s * s;
    double t = 1.0 / 21.0;
    t = fma(t, z, 1.0 / 19.0); t = fma(t, z, 1.0 / 17.0); t = fma(t, z, 1.0 / 15.0); t = fma(t, z, 1.0 / 13.0);
    t = fma(t, z, 1.0 / 11.0); t = fma(t, z, 1.0 / 9.0); t = fma(t, z, 1.0 / 7.0); t = fma(t, z, 0.2); t = fma(t, z, 1.0 / 3.0);
    const double lm = fma(s * z, t, s);                               // atanh(s)
    return -fma((double)e, 0.30102999566398119521, lm * 0.86858896380650365530);   // log10(2), 2 / ln(10)
}
__device__ __forceinline__ double neg_log10_1m(double p) {              // smCounter.py:509-510
    const double x = 1.0 - p;
    if (!(x > 0.0)) return 16.0;
    if (x < 2.2250738585072014e-308) return -log10(x);                  // subnormal: library call
    return neg_log10_normal(x);
}

// -log10(x) for x = fl(1 - p) when p is tiny: with q = 1 - x (exact, Sterbenz) the series q + q^2/2 + ... + q^6/6 is within
// 2e-16 relative of -ln(x) for q < 2^-10, so the result agrees with log10(x) to the last bit or two -- and it costs a
// sixth of the library call.  (The posterior of a padded allele is ~1e-5: every barcode takes this branch once.)
__device__ __forceinline__ double neg_log10_1m_small(double p) {
    const double x = 1.0 - p;
    const double q = 1.0 - x;
    if (!(q < 0.0009765625)) return neg_log10_1m(p);
    double s = fma(q, 1.0 / 6.0, 0.2);
    s = fma(s, q, 0.25);
    s = fma(s, q, 1.0 / 3.0);
    s = fma(s, q, 0.5);
    s = fma(s, q, 1.0);
    return (s * q) * 0.43429448190325182765;             // 1 / ln(10)
}

// MTCnt / strongMTCnt of an allele that may be dynamic, straight to the per-locus accumulators
__device__ __forceinline__ void bump_mt_global(int32_t* cnt, size_t nl, int64_t L, int32_t* dcnt, uint32_t aid, bool strong) {
    int32_t* row = aid < NF ? cnt + (size_t)aid * SMC_NCNT * nl + L : dcnt + (size_t)(aid - NF) * SMC_NCNT;
    const size_t stride = aid < NF ? nl : 1;
    atomicAdd(&row[SMC_C_MT * stride], 1);
    if (strong) atomicAdd(&row[SMC_C_STRONG * stride], 1);
}

// calProb + consensus for a barcode that shows several alleles, a DEL / dynamic allele, or more fragments than the prior
// table holds (smCounter.py:26-98, 506-523) -- the general form, for the barcode U at locus L; its PI terms and MT counts go
// to the per-locus accumulators with atomics.  Returns the finalDict keys it touched among the fixed alleles.
__device__ __noinline__ uint32_t umi_general(DynTab T, const double* __restrict__ pcrtab, int pcr_nmax, double smt,
                                             int32_t* cnt, unsigned long long* limb, size_t nl, int64_t L, UmiState& U) {
    const int n = U.n, ndyn = U.ndyn;
    const double rightP = U.rightP;
    uint32_t exist = U.exist, keymask = 0;
    // canonical order of the dynamic slots = ascending allele key (insertion sort of the slot rows; a slot whose exist bit is
    // clear -- its fragments were all deleted again -- travels with its bit)
    for (int i = 1; i < ndyn; ++i)
        for (int j = i; j > 0 && __ldcg(&T.dkey[U.dyn[j - 1]]) > __ldcg(&T.dkey[U.dyn[j]]); --j) {
            const int a = NF + j - 1, b = NF + j;
            const uint32_t tu = U.dyn[j - 1]; U.dyn[j - 1] = U.dyn[j]; U.dyn[j] = tu;
            const int tc = U.cnt[a]; U.cnt[a] = U.cnt[b]; U.cnt[b] = tc;
            const double tp = U.prod[a]; U.prod[a] = U.prod[b]; U.prod[b] = tp;
            const uint32_t ba = (exist >> a) & 1u, bb = (exist >> b) & 1u;
            exist = (exist & ~((1u << a) | (1u << b))) | (bb << a) | (ba << b);
        }
    int k = __popc(exist);
    uint32_t pad = 0;                             // :49-54  pad with A, T, G, C until 4
    if (k < 4 && !((exist >> SMC_A_A) & 1u)) { pad |= 1u << SMC_A_A; ++k; }
    if (k < 4 && !((exist >> SMC_A_T) & 1u)) { pad |= 1u << SMC_A_T; ++k; }
    if (k < 4 && !((exist >> SMC_A_G) & 1u)) { pad |= 1u << SMC_A_G; ++k; }
    if (k < 4 && !((exist >> SMC_A_C) & 1u)) { pad |= 1u << SMC_A_C; ++k; }
    const uint32_t uniq = exist | pad;
    const double INF = __longlong_as_double(0x7ff0000000000000ll);
    // ---- PCR prior of every allele of the barcode (:79-81): table lookups (host glibc pow) or pow()
    const bool tab = (k <= 6 && n <= pcr_nmax);
    const double* trow = pcrtab + ((size_t)(k - 4) * ((size_t)(pcr_nmax + 1) * (pcr_nmax + 2) / 2) + (size_t)n * (n + 1) / 2);
    const double denom = (double)n + 0.5 * (double)k;
    const double pcr_pad = tab ? __ldg(trow) : pcr_slow(0, denom);
    double m1 = pad ? pcr_pad : INF, m2 = INF; int arg1 = -1;      // smallest / second smallest prior and its slot
    double tpad = rightP;                                         // :88-91
    for (uint32_t m = exist; m; m &= m - 1) {
        const int s = __ffs(m) - 1;
        const int c = U.cnt[s];
        const double v = tab ? __ldg(trow + c) : pcr_slow(c, denom);
        tpad = __dmul_rn(tpad, v);
        if (v < m1) { m2 = m1; m1 = v; arg1 = s; } else if (v < m2) m2 = v;
    }
    // ---- likelihood of each present allele (:86), stored over its (no longer needed) product; pads all share tpad
    const double PCR_NO_ERROR = 1.0 - 3e-5;                       // smCounter.py:20
    for (uint32_t m = exist; m; m &= m - 1) {
        const int s = __ffs(m) - 1;
        const double minp = (s == arg1) ? m2 : m1;                // min over the OTHER members of uniq
        U.prod[s] = __dadd_rn(__dmul_rn(PCR_NO_ERROR, U.prod[s]), __dmul_rn(rightP, minp));
    }
    double sumP = 0.0;                                            // :93, in canonical slot order
    for (uint32_t m = uniq; m; m &= m - 1) {
        const int s = __ffs(m) - 1;
        sumP = __dadd_rn(sumP, ((exist >> s) & 1u) ? U.prod[s] : tpad);
    }
    // ---- posterior -> -log10(1-p) (:96, :509-510), PI accumulation (:512), consensus (:514-523).
    // One loop over the members of uniq in slot order; the pads share one value (computed at the first pad).
    double best = -1.0, l_pad = 0.0; int nbest = 0, cons = -1; bool have_pad = false;
    unsigned long long plo = 0, phi = 0;
#pragma unroll 1
    for (uint32_t m = uniq; m; m &= m - 1) {
        const int s = __ffs(m) - 1;
        const bool is_pad = (pad >> s) & 1u;
        double l; unsigned long long lo, hi;
        if (is_pad && have_pad) { l = l_pad; lo = plo; hi = phi; }
        else {
            l = neg_log10_1m(sumP <= 0.0 ? 0.0 : (is_pad ? tpad : U.prod[s]) / sumP);
            pi_fixed128(l, lo, hi);
            if (is_pad) { have_pad = true; l_pad = l; plo = lo; phi = hi; }
        }
        if (s < NF) {
            add_limbs(limb + (size_t)s * 3 * nl + L, nl, lo, hi);
            keymask |= 1u << s;
        } else {
            const uint32_t e = U.dyn[s - NF];
            add_limbs(T.dlimb + (size_t)e * 3, 1, lo, hi);
            T.diskey[e] = 1;
        }
        if (l > best) { best = l; nbest = 1; cons = s; }
        else if (l == best) nbest++;
    }
    if (nbest == 1) {                                             // :515-519
        const uint32_t aid = cons < NF ? (uint32_t)cons : NF + U.dyn[cons - NF];
        bump_mt_global(cnt, nl, L, T.dcnt, aid, best > smt);
    } else if (n == 1) {                                          // :521-523
        bump_mt_global(cnt, nl, L, T.dcnt, U.last_aid, false);
    }
    return keymask;
}

// down-sampling mask / barcode listing for the barcode that closes (both rare: only loci with more barcodes than ds)
struct MaskListArgs {        // by value: taking the address of the kernel parameter block would copy it to local memory
    const int64_t* keep_off; const uint64_t* keep_umi; const uint64_t* umi_of_urank;
    uint32_t* list_count; const int64_t* list_off; uint64_t* list_umi; uint32_t* list_first; int64_t list_cap;
};
template <bool LIST>
__device__ __noinline__ bool umi_mask_and_list(MaskListArgs A, int ki, int li, uint32_t urank, uint32_t first_read) {
    bool used = true;
    const unsigned long long u = A.umi_of_urank[urank];
    if (ki >= 0) {                                   // smCounter.py:496-500
        int64_t lo = A.keep_off[ki], hi = A.keep_off[ki + 1];
        int64_t pos = lower_bound_u64((const uint64_t*)A.keep_umi + lo, hi - lo, u);
        used = (pos < hi - lo) && (A.keep_umi[lo + pos] == u);
    }
    if (LIST && li >= 0) {
        uint32_t slot = atomicAdd(&A.list_count[li], 1u);
        int64_t o = A.list_off[li] + slot;
        if (o < A.list_off[li + 1] && o < A.list_cap) { A.list_umi[o] = u; A.list_first[o] = first_read; }
    }
    return used;
}

// calProb + the per-barcode part of vc() (smCounter.py:26-98, 506-532) for the lane's locus; the general form of calProb is
// deferred: `rec` is the record k_merge_deferred gets for it.
template <bool LIST>
__device__ __forceinline__ void umi_finalize(const KBArgs& A, int lane, int ki, int li, uint32_t umi_slot, uint4 rec, int* fc, ulonglong2* limb,
                                             MergeState& S) {
    if (S.flags & LF_UMI_SEEN) S.allMT++;
    bool used = S.flags & LF_UMI_BC;
    if (used) {
        S.nBC++;
        if (ki >= 0 || (LIST && li >= 0)) {
            MaskListArgs M;
            M.keep_off = A.keep_off; M.keep_umi = A.keep_umi; M.umi_of_urank = A.umi_of_urank; M.list_count = A.list_count;
            M.list_off = A.list_off; M.list_umi = A.list_umi; M.list_first = A.list_first; M.list_cap = A.list_cap;
            used = umi_mask_and_list<LIST>(M, ki, li, A.umi_urank[umi_slot], S.first_read);
        }
    }
    if (used) {
        const int n = S.n;
        S.usedMT++; S.usedFrag += n;
        S.mt3 += n >= 3; S.mt5 += n >= 5; S.mt7 += n >= 7; S.mt10 += n >= 10;
        const uint32_t ACGT = (1u << SMC_A_A) | (1u << SMC_A_T) | (1u << SMC_A_G) | (1u << SMC_A_C);
        if (n <= A.mtDrop) {                              // :28-32 -> four zeros, a 4-way tie (:514-523)
            S.keymask |= ACGT;
            if (n == 1) bump_mt(A.T.dcnt, fc, lane, S.last_aid, 1u);
        } else if (!(S.flags & LF_DEFER) && (S.exist & ACGT) && n <= A.pcr_nmax) {
            // ---- fast path: every fragment of the barcode shows the same base a0 in {A,C,G,T}; uniq = {A,C,G,T} (:49-54).
            // Same operations in the same order as umi_general (prodP[a0] == rightP, one present allele, three pads
            // sharing one value), with all intermediates in registers.
            const int a0 = __ffs(S.exist) - 1;
            const double rightP = S.rightP;
            const double* trow = A.pcrtab + (size_t)n * (n + 1) / 2;                       // k = 4
            const double v_e = __ldg(trow + n), v_pad = __ldg(trow);                       // :79-81
            const double tpad = __dmul_rn(rightP, v_e);                                    // :88-91
            const double PCR_NO_ERROR = 1.0 - 3e-5;
            const double t_e = __dadd_rn(__dmul_rn(PCR_NO_ERROR, rightP), __dmul_rn(rightP, v_pad));   // :86 (min over the others = a pad's prior)
            const int posidx = a0 - (a0 > SMC_A_DEL ? 1 : 0);                              // rank of a0 in slot order A C T G
            double sumP = posidx == 0 ? t_e : tpad;                                        // :93 (0.0 + x == x)
            sumP = __dadd_rn(sumP, posidx == 1 ? t_e : tpad);
            sumP = __dadd_rn(sumP, posidx == 2 ? t_e : tpad);
            sumP = __dadd_rn(sumP, posidx == 3 ? t_e : tpad);
            const bool pos = sumP > 0.0;
            const double l_pad = neg_log10_1m_small(pos ? tpad / sumP : 0.0);              // :96, :509-510
            const double l_e = neg_log10_1m(pos ? t_e / sumP : 0.0);
            // PI: l_pad goes to all four bases through the register accumulator, a0 gets the difference (mod 2^128)
            unsigned long long plo, phi, elo, ehi;
            pi_fixed128(l_pad, plo, phi);
            pi_fixed128(l_e, elo, ehi);
            add128(S.pad_lo, S.pad_hi, plo, phi);
            sub128(elo, ehi, plo, phi);
            ulonglong2 v = LIMB(a0);
            add128(v.x, v.y, elo, ehi);
            LIMB(a0) = v;
            S.keymask |= ACGT;
            // consensus (:514-523): three pads tie at l_pad; a0 wins iff l_e > l_pad
            if (l_e > l_pad) FCW(a0) += (l_e > A.smt) ? 0x10001 : 1;
            else if (n == 1) FCW(a0) += 1;
        } else {
            rec.w &= ~DR_STATUS_ONLY;
        }
    }
    // the general form, or a deferred barcode outside the call that may hold more dynamic alleles than its slots
    if (!(rec.w & DR_STATUS_ONLY) || ((S.flags & LF_DEFER) && S.n > NDYN)) {
        const uint32_t r = atomicAdd(A.defer_count, 1u);
        if (r < A.defer_cap) A.defer[r] = rec;
        else atomicOr(A.T.gflags, GF_DEFER_FULL);
    }
    S.n = 0; S.exist = 0; S.rightP = 1.0; S.flags = 0; S.first_read = 0xffffffffu;
}

template <bool LIST>
__global__ void __launch_bounds__(KB_WARPS * 32, KB_MINBLOCKS) k_merge_t(const KBArgs A) {
    extern __shared__ __align__(16) uint32_t smem[];
    double* q_s = reinterpret_cast<double*>(smem);           // complement of the fragment probability (smCounter.py:65-68, :77)
    for (int i = threadIdx.x; i < 257; i += KB_WARPS * 32) q_s[i] = 1.0 - (i == 0 ? 0.1 : __ldg(&A.bqtab[i - 1]));
    __syncthreads();
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t* ws = smem + KB_TAB_BYTES / 4 + (size_t)w * KB_WARP_WORDS;
    int* fc = (int*)ws;
    ulonglong2* limb = (ulonglong2*)(ws + KB_FC_WORDS);

    const uint32_t unit = A.unit0 + blockIdx.x * KB_WARPS + w;
    if (unit >= A.n_units) return;
    const uint32_t F = A.unit_nfrag[unit];
    if (F == 0) return;
    const uint32_t eb = A.unit_eb[unit], ee = A.unit_ee[unit];
    const uint32_t tile = A.unit_tile[unit];
    const uint64_t so = unit_slot_base(eb, unit, A.code_mult);
    const uint32_t cap = unit_slot_cap(ee - eb, A.code_mult);

    const int64_t L = (int64_t)tile * 32 + lane;
    const bool lane_valid = L < A.n_loci;
    const int ki = (lane_valid && A.keep_idx) ? A.keep_idx[L] : -1;
    const int li = (LIST && lane_valid) ? A.list_idx[L] : -1;

    for (int i = lane; i < KB_FC_WORDS + KB_LIMB_WORDS; i += 32) ws[i] = 0;
    __syncwarp();

    MergeState S;
    S.allFrag = S.allMT = S.usedFrag = S.nBC = S.usedMT = S.mt3 = S.mt5 = S.mt7 = S.mt10 = 0;
    S.keymask = 0; S.pad_lo = S.pad_hi = 0;
    S.flags = 0;
    S.n = 0; S.exist = 0; S.rightP = 1.0; S.last_aid = 0;
    S.first_read = 0xffffffffu;

    // warp uniform: umi_urank[] slot, first fragment code and the extension rows before it of the open barcode; rows read
    uint32_t umi_slot = eb, umi_f = 0, umi_x = 0, nx = 0;
    const uint4* cp = A.codes + (so >> 3) * 32 + lane;
    const uint32_t* extp = reinterpret_cast<const uint32_t*>(A.codes) + (so + cap) * 16 + lane;   // extension rows, downward
    const uint32_t* ffp = LIST ? A.frag_first + so * 32 + lane : nullptr;
    uint4 v = __ldg(cp), vn = v;
    // One pass over the F fragment codes plus a virtual "next barcode" code that closes the last barcode: a single
    // umi_finalize site keeps the loop small in the instruction cache.
#pragma unroll 1
    for (uint32_t f = 0; f <= F; ++f) {
        if ((f & 7u) == 0u) {
            v = vn;
            cp += 32;
            if (f + 8u < F) vn = __ldg(cp);                            // prefetch the next group of eight
        }
        const uint32_t cd = f < F ? (v.x & 0xffffu) : FC_UMIFIRST;
        v.x = __funnelshift_r(v.x, v.y, 16); v.y = __funnelshift_r(v.y, v.z, 16); v.z = __funnelshift_r(v.z, v.w, 16); v.w >>= 16;
        if (cd & FC_UMIFIRST) {                                        // warp uniform
            if (f != 0u) {                                             // the previous barcode is complete
                umi_finalize<LIST>(A, lane, ki, li, umi_slot, make_uint4(unit, umi_f, umi_x, (uint32_t)lane | DR_STATUS_ONLY), fc, limb, S);
                ++umi_slot;
            }
            umi_f = f; umi_x = nx;
        }
        const uint32_t st = (cd >> FC_ST_SH) & 3u;
        S.allFrag += st ? 1 : 0;                                       // :463-464
        S.flags |= (st ? LF_UMI_SEEN : 0u) | (st & LF_UMI_BC);         // st >= 2: the barcode is a key of bcDict
        if (LIST) { S.first_read = min(S.first_read, f < F ? __ldg(ffp) : 0xffffffffu); ffp += 32; }
        uint32_t aid = (cd >> FC_AID_SH) & 7u;
        if (cd & FC_EXT) {                                             // warp uniform
            extp -= 32; ++nx;
            const uint32_t e = __ldg(extp);
            if (aid == FC_AID_DYN) aid = NF + e;
        }
        const double q = q_s[((cd >> 13) & 1u) * ((cd & 0xffu) + 1u)];                  // smCounter.py:65-68 (a valid entry for any code)
        const bool join = st == 3u;
        // The fragment joins a barcode that has shown one allele so far (fragment_join reduces to a product and a count),
        // branch free -- a fragment that is not in bcDict multiplies by exactly 1.0.  A second allele or a dynamic one defers
        // the barcode to k_merge_deferred; from then on only its count and last allele matter here.
        const uint32_t bit = 1u << (aid & 31u);
        S.flags |= (join && (aid >= NF || (S.exist & ~bit) != 0u)) ? LF_DEFER : 0u;
        S.rightP = __dmul_rn(S.rightP, join ? q : 1.0);                                  // :77
        S.n += join ? 1 : 0;
        S.exist |= join ? bit : 0u;
        S.last_aid = join ? aid : S.last_aid;
    }
    // ---- flush the lane's locus to the per-locus accumulators ([field][locus] layout: coalesced across lanes)
    if (lane_valid) {
        const size_t nl = (size_t)A.n_loci;
#pragma unroll
        for (int a = 0; a < NF; ++a) {
            const uint32_t mv = (uint32_t)FCW(a);
            if (mv & 0xffffu) atomicAdd(&A.cnt[((size_t)a * SMC_NCNT + SMC_C_MT) * nl + L], (int)(mv & 0xffffu));
            if (mv >> 16) atomicAdd(&A.cnt[((size_t)a * SMC_NCNT + SMC_C_STRONG) * nl + L], (int)(mv >> 16));
            ulonglong2 v2 = LIMB(a);
            if (a != SMC_A_DEL) add128(v2.x, v2.y, S.pad_lo, S.pad_hi);
            add_limbs(A.limb + (size_t)a * 3 * nl + L, nl, v2.x, v2.y);
        }
        int32_t* loc = A.loc;
        if (S.allFrag) atomicAdd(&loc[SMC_L_ALLFRAG * nl + L], S.allFrag);
        if (S.allMT) atomicAdd(&loc[SMC_L_ALLMT * nl + L], S.allMT);
        if (S.usedFrag) atomicAdd(&loc[SMC_L_USEDFRAG * nl + L], S.usedFrag);
        if (S.nBC) atomicAdd(&loc[SMC_L_NBC * nl + L], S.nBC);
        if (S.usedMT) atomicAdd(&loc[SMC_L_USEDMT * nl + L], S.usedMT);
        if (S.mt3) atomicAdd(&loc[SMC_L_MT3 * nl + L], S.mt3);
        if (S.mt5) atomicAdd(&loc[SMC_L_MT5 * nl + L], S.mt5);
        if (S.mt7) atomicAdd(&loc[SMC_L_MT7 * nl + L], S.mt7);
        if (S.mt10) atomicAdd(&loc[SMC_L_MT10 * nl + L], S.mt10);
        if (S.keymask) atomicOr(&loc[SMC_L_KEYMASK * nl + L], (int)S.keymask);
    }
}

// The barcodes k_merge deferred, one thread per record: the barcode's fragments at the lane's locus run through the general
// fragment_join again, from its first fragment code to the next barcode's, and umi_general finishes it.  Every fragment takes
// the same operations in the same order as it would have inside k_merge; the results go to the same accumulators with atomics
// (integers and 128-bit fixed point, so where and when they are added does not change them).
__global__ void __launch_bounds__(KD_THREADS) k_merge_deferred(const KBArgs A) {
    const uint32_t nrec = min(*A.defer_count, A.defer_cap);
    const size_t nl = (size_t)A.n_loci;
    for (uint32_t r = blockIdx.x * KD_THREADS + threadIdx.x; r < nrec; r += gridDim.x * KD_THREADS) {
        const uint4 rec = A.defer[r];
        const uint32_t unit = rec.x, lane = rec.w & 31u;
        const uint32_t F = A.unit_nfrag[unit], eb = A.unit_eb[unit], ee = A.unit_ee[unit];
        const uint64_t so = unit_slot_base(eb, unit, A.code_mult);
        const uint32_t cap = unit_slot_cap(ee - eb, A.code_mult);
        const int64_t L = (int64_t)A.unit_tile[unit] * 32 + lane;
        const uint16_t* cp = reinterpret_cast<const uint16_t*>(A.codes) + so * 32 + lane * 8;      // code f: cp[(f >> 3) * 256 + (f & 7)]
        const uint32_t* extp = reinterpret_cast<const uint32_t*>(A.codes) + (so + cap) * 16 + lane - (size_t)rec.z * 32;
        UmiState U;
        U.n = 0; U.exist = 0; U.Q = 1.0; U.rightP = 1.0; U.last_aid = 0; U.ndyn = 0; U.status = 0;
#pragma unroll 1
        for (uint32_t f = rec.y; f < F; ++f) {
            const uint32_t cd = __ldg(cp + (f >> 3) * 256 + (f & 7u));
            if ((cd & FC_UMIFIRST) && f != rec.y) break;
            uint32_t aid = (cd >> FC_AID_SH) & 7u;
            if (cd & FC_EXT) {
                extp -= 32;
                const uint32_t e = __ldg(extp);
                if (aid == FC_AID_DYN) aid = NF + e;
            }
            if (((cd >> FC_ST_SH) & 3u) == 3u) {
                const uint32_t i = ((cd >> 13) & 1u) * ((cd & 0xffu) + 1u);                   // as k_merge's table
                const double pf = i == 0 ? 0.1 : __ldg(&A.bqtab[i - 1]);
                fragment_join(pf, 1.0 - pf, aid, U);
            }
        }
        if (U.status) atomicOr(&A.loc[SMC_L_STATUS * nl + L], (int)U.status);
        if (rec.w & DR_STATUS_ONLY) continue;
        if (U.exist && !(U.exist & (U.exist - 1u))) umi_fill_single(U);      // a DEL, or more fragments than the prior table holds
        const uint32_t keymask = umi_general(A.T, A.pcrtab, A.pcr_nmax, A.smt, A.cnt, A.limb, nl, L, U);
        if (keymask) atomicOr(&A.loc[SMC_L_KEYMASK * nl + L], (int)keymask);
    }
}
