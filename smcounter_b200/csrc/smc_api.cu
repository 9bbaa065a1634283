// libsmc_b200.so -- C ABI (include/smc_b200.h) and pipeline orchestration.
//
//   H2D (scalars first; bases / qualities in chunks on a second stream, overlapped with everything up to K3)
//       -> K2a barcode slots (hash table) + one radix sort of the fragment ids on barcode slot     smc_sort.cuh
//       -> K1 read prep (CIGAR walk, QC gate, locus range, stored window)                         smc_pileup.cuh
//       -> K2b (read x 32-locus tile) events, radix sort by tile                                  smc_sort.cuh
//       -> K3a k_gather: lane = locus, base/quality gather, read tallies, fragment merge smc_pileup.cuh
//          (bases and qualities expanded per chunk into one 16-bit word per stored base first)     smc_upload.cuh
//       -> K3b k_merge: per-barcode posterior (calProb), prediction index, consensus    smc_pileup.cuh
//          (k_merge_deferred: the barcodes whose calProb takes the general form)
//       -> K4 FP64 statistics: PI, ALT, filters, Fisher                                smc_stats.cuh
//       -> (SMC_DS_DEVICE, loci flagged for down-sampling only) listing pass, Py2 draw, K3 + K4 again with the drawn masks
//                                                                                      smc_downsample.cuh
//   -> D2H
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <new>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include <nvtx3/nvToolsExt.h>      // header-only: ranges show up under nsys / ncu --nvtx, cost nothing otherwise

#include "smc_common.cuh"
#include "smc_sort.cuh"
#include "smc_pileup.cuh"
#include "smc_stats.cuh"
#include "smc_upload.cuh"
#include "smc_downsample.cuh"
#include "smc_bgzf.cuh"

namespace {

// NVTX range over one pipeline stage (SURVEY.md section 5: tracing)
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

thread_local std::string g_create_error;
// Contexts of one process that upload to the same GPU take turns on the host link: the chunked copies of a batch start
// after those of the batch enqueued before it (an event at the tail of each context's copies).  Two copy streams running
// side by side would each get half the link, finish together and leave the GPU idle until then; in turns, the first
// batch's kernels start while the second one is still arriving.  SMC_LINK_TURNS=0 switches it off.
static std::mutex g_link_mu;
static cudaEvent_t g_link_tail[64] = {};
static smc_ctx* g_link_owner[64] = {};

// Device scratch, grown lazily.  Stream-ordered allocations from the device's default memory pool (its release threshold
// is raised in smc_ctx_create): growing a buffer or destroying a context hands the memory back to the pool, not to the
// driver, so the next batch / the next context of the process does not pay cudaMalloc / cudaFree again (measured: a fresh
// context right after another one was destroyed spent 100-900 ms in cudaMalloc for a 0.3 M read batch).
// Every buffer joins its context's registry when it is constructed: the context gives it its stream and releases it.
struct DevBuf {
    void* p = nullptr; size_t cap = 0; cudaStream_t st = nullptr;
    explicit DevBuf(std::vector<DevBuf*>& registry) { registry.push_back(this); }
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFreeAsync(p, st);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMallocAsync(&p, want, st);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFreeAsync(p, st); p = nullptr; cap = 0; }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

}  // namespace

#define PCR_NMAX 192

// words of the small device scratch block (smc_ctx::d_small) the kernels report through
enum SmallWord {
    SW_FRAG_OR = 0,          // u64: OR of the fragment ids k_umi_slots found out of range (0: all ids are dense)
    SW_N_TILE_EVENTS = 4,    // total of the tile-event scan
    SW_GFLAGS = 5,           // GF_* bits raised by the kernels
    SW_DYN_COUNT = 6,        // entries of the dynamic-allele table
    SW_N_TASKS = 7,          // Fisher tasks emitted by k_call
    SW_CVG_SUM = 8,          // u64: sum of cvg over the loci (= pileup read-events)
    SW_N_MULTI = 10,         // reads of fragments of >= 3 reads (k_place_reads)
    SW_N_UMI = 12,           // distinct barcodes (k_frag_scan)
    SW_DS_LOCI = 13,         // loci k_call flagged SMC_ST_NEED_DOWNSAMPLE (device draw on), then u64 at 14: their barcodes
    SW_PIPE_BLOCKED = 16,    // [SMC_PIPE_MAX]: first unit that has to wait for chunk c + 1
    SW_PACK_TOTALS = 40,     // [6]: bytes / words of packed bases, qualities, CIGARs, compact qualities, compact bases; bq[] words
    SW_DEFER_COUNT = 48,     // deferred-barcode records k_merge appended
    SW_DS_MISSING = 50,      // u64: a dictionary-coded barcode of a drawn locus that has no hash (0: none)
    SW_DS_OR = 52,           // u64: OR of the barcode codes of the drawn loci
    SW_CHUNK_FIRST = 64      // [SMC_PIPE_MAX]: k_chunk_need's first read per upload chunk
};

// stage events of ctx->ev; the SMC_TIMELINE line prints the first seven, in this order
enum StageEvent {
    EV_COPY_BEGIN, EV_COPY_END,                 // host link: the upload (H2D), or smc_download (D2H)
    EV_RUN_BEGIN, EV_PREP_DONE, EV_SORT_DONE, EV_PILEUP_DONE, EV_STATS_DONE,
    EV_PILEUP_BEGIN, EV_GATHER_DONE, EV_MERGE_DONE,
    EV_READ_SORT_BEGIN, EV_READ_SORT_DONE, EV_READ_PREP_BEGIN, EV_READ_PREP_DONE, EV_EVENT_SORT_BEGIN, EV_EVENT_SORT_DONE,
    EV_COUNT
};

struct smc_ctx {
    int device = 0;
    smc_params prm{};
    std::string err;
    cudaStream_t st = nullptr;
    cudaEvent_t ev[EV_COUNT]{};
    std::vector<DevBuf*> bufs;                  // every DevBuf member below (DevBuf's constructor)
    // pipelined upload of smc_call_batch: bases / qualities arrive in chunks on st_copy while st already computes
    cudaStream_t st_copy = nullptr;
    cudaEvent_t ev_link = nullptr, ev_tmp = nullptr, ev_tmp2 = nullptr, ev_chunk[SMC_PIPE_MAX]{};
    int pipe_n = 0;                             // > 1: the chunk events of the current batch are pending / recorded
    DevBuf d_pipe_need{bufs};
    bool packed_seq = false, packed_qual = false, packed_cigar = false;   // offsets were NULL: computed on the device
    uint32_t pipe_end[SMC_PIPE_MAX]{};          // launch c of the pileup kernels covers units [pipe_end[c-1], pipe_end[c])
    // resident inputs
    int64_t n_reads = 0, n_loci = 0;
    int64_t seq_bytes = 0, qual_bytes = 0, n_cigar_words = 0;
    DevBuf d_ref_id{bufs}, d_pos{bufs}, d_flag{bufs}, d_mapq{bufs}, d_nm{bufs}, d_lseq{bufs}, d_cig_off{bufs}, d_ncig{bufs}, d_umi{bufs},
        d_frag{bufs}, d_cigar{bufs}, d_store_lo{bufs}, d_store_len{bufs};
    bool has_store = false;                     // reads carry a stored window (smc_reads_soa::store_lo / store_len)
    // Bases and qualities as uploaded (d_seq_up / d_qual_up, any encoding; byte offsets per read in d_seq_poff / d_qual_poff,
    // narrowed from the caller's d_seq_off / d_qual_off when it gives them) are expanded into the one array the kernels read:
    // bq[], quality | BAM nibble << 8 per stored base, d_bq_off the word of each read's first stored base
    int qual_bits = 8, seq_bits = 4; int64_t n_seq_exc = 0;
    DevBuf d_seq_up{bufs}, d_qual_up{bufs}, d_seq_off{bufs}, d_qual_off{bufs}, d_seq_poff{bufs}, d_qual_poff{bufs}, d_qual_lut{bufs},
        d_exc_read{bufs}, d_exc_pos{bufs}, d_exc_nib{bufs}, d_bq{bufs}, d_bq_off{bufs}, d_stage{bufs}, d_defer{bufs};
    uint32_t bq_cap = 0;                        // words of d_bq the current batch may fill
    uint32_t defer_cap = 0;                     // records in the deferred-barcode list of k_merge (grows x4 on GF_DEFER_FULL)
    DevBuf d_loci_ref{bufs}, d_loci_pos{bufs}, d_loci_base{bufs}, d_loci_key{bufs};
    DevBuf d_keep_idx{bufs}, d_keep_off{bufs}, d_keep_umi{bufs};
    bool has_keep = false, uploaded = false, ran = false;
    // tables
    DevBuf d_bqtab{bufs}, d_pcrtab{bufs};
    // scratch
    DevBuf d_k0{bufs}, d_k1{bufs}, d_v0{bufs}, d_v1{bufs}, d_hist{bufs}, d_scan{bufs}, d_urank{bufs}, d_frank{bufs}, d_umi_of_urank{bufs},
        d_recs{bufs}, d_ek0{bufs}, d_ek1{bufs}, d_ev0{bufs}, d_ev1{bufs}, d_tile_off{bufs}, d_unit_cnt{bufs}, d_unit_off{bufs}, d_small{bufs},
        d_grec{bufs}, d_unit_eb{bufs}, d_unit_ee{bufs}, d_unit_tile{bufs}, d_unit_nfrag{bufs}, d_codes{bufs}, d_frag_first{bufs},
        d_umi_urank{bufs}, d_umi_table{bufs}, d_frag_cnt{bufs}, d_frag_min{bufs};
    uint32_t code_mult = 1;                     // fragment-code storage per tile event (1, or 3 = worst case after GF_CODE_FULL)
    uint32_t n_units_cap = 0;
    // per-locus accumulators / outputs
    DevBuf d_loc{bufs}, d_cnt{bufs}, d_limb{bufs}, d_pi{bufs}, d_max{bufs}, d_second{bufs}, d_alt{bufs}, d_altpi{bufs}, d_secondpi{bufs},
        d_fl1{bufs}, d_fl2{bufs}, d_bial{bufs}, d_fp{bufs}, d_for{bufs};
    // dynamic allele table + sorted rows
    uint32_t dyn_cap = 0;
    DevBuf d_dkey{bufs}, d_drep_read{bufs}, d_drep_qpos{bufs}, d_dlen{bufs}, d_dcnt{bufs}, d_dlimb{bufs}, d_diskey{bufs};
    DevBuf d_lk0{bufs}, d_lv0{bufs}, d_lv1{bufs};
    DevBuf d_s_key{bufs}, d_s_cnt{bufs}, d_s_limb{bufs}, d_s_iskey{bufs}, d_s_pi{bufs}, d_s_rep_read{bufs}, d_s_rep_qpos{bufs}, d_s_len{bufs},
        d_dyn_first{bufs};
    int64_t n_dyn = 0;
    DevBuf d_tasks{bufs};
    uint32_t task_cap = 0;
    // barcode listing
    DevBuf d_list_idx{bufs}, d_list_count{bufs}, d_list_off{bufs}, d_list_umi{bufs}, d_list_first{bufs};
    DevBuf d_hp_bases{bufs}, d_hp_meta{bufs}, d_hp_flags{bufs};     // smc_hp_lowcomp
    // down-sampling drawn on the device (smc_set_downsample): the flagged loci of the last call_stats, the caller's part of the
    // mask CSR, the keep index from which masks were drawn, the Py2 hashes of dictionary-coded barcodes, and the draw's scratch
    int ds_mode = SMC_DS_FLAG;
    int64_t ds_flagged = 0, ds_barcodes = 0;
    int64_t keep_n = 0, keep_total = 0;
    int32_t ds_first_drawn = INT32_MAX;
    int64_t n_bc = 0;
    DevBuf d_bc_code{bufs}, d_bc_hash{bufs};
    DevBuf d_ds_flag{bufs}, d_ds_nbc{bufs}, d_ds_locus{bufs}, d_ds_k0{bufs}, d_ds_k1{bufs}, d_ds_v0{bufs}, d_ds_v1{bufs}, d_ds_codes{bufs},
        d_ds_hash{bufs}, d_ds_scratch{bufs}, d_ds_keep_off{bufs}, d_ds_keep_umi{bufs};
    // BAM decode (smc_decode_bam): device passes, and the decoded arrays in one pinned host arena owned by the context
    DevBuf d_bz_comp{bufs}, d_bz_jobs{bufs}, d_bz_raw{bufs}, d_bz_scratch{bufs}, d_bz_status{bufs}, d_bz_walk{bufs}, d_bz_base{bufs},
        d_bz_offs{bufs}, d_bz_info{bufs}, d_bz_cnt{bufs}, d_bz_k0{bufs}, d_bz_k1{bufs}, d_bz_v0{bufs}, d_bz_v1{bufs}, d_bz_first{bufs},
        d_bz_isfirst{bufs}, d_bz_dfirst{bufs}, d_bz_disfirst{bufs}, d_bz_hist{bufs}, d_bz_scan{bufs}, d_bz_tg{bufs}, d_bz_out{bufs},
        d_bz_dict{bufs}, d_bz_small{bufs};
    void* h_bz_out = nullptr; size_t h_bz_cap = 0;
    int n_sm = 148;                             // multiprocessors of the device (smc_ctx_create)
    std::vector<std::string> bz_dict;
    uint64_t* bz_qual_hist = nullptr;
    smc_timings tm{};
    uint32_t chunk = 128;       // tile events per warp unit (A/B on B200, whole step: 96 -> 4.42 ms, 128 -> 4.39, 160 -> 4.39, 256 -> 4.47, 384 -> 4.60)
    const uint32_t* ev_read_sorted = nullptr;   // tile-sorted event -> srank map (lives in d_ev0 or d_ev1)
    int64_t n_tile_events = 0;
    int64_t ne_cap = 0;                         // capacity of the tile-event buffers (grow only)
};

#define CK(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e__ = (call);                                                                        \
        if (e__ != cudaSuccess) {                                                                        \
            ctx->err = std::string(#call) + ": " + cudaGetErrorString(e__);                              \
            return SMC_E_CUDA;                                                                           \
        }                                                                                                \
    } while (0)

// ------------------------------------------------------------------------------------------------------------
// small kernels used only by the orchestration
// ------------------------------------------------------------------------------------------------------------
// Barcode slots and per-fragment facts.  Every distinct barcode code gets one slot of an open-addressing table (linear probing,
// atomicCAS); the slot index stands in for the barcode in the fragment sort key.  Which slot a barcode lands in may differ from
// run to run; nothing downstream depends on the order of barcodes (the PI sums are fixed point, every other accumulation is an
// integer).  The last slot (mask) is never handed out: FRAG_NONE, the key of fragment ids no read carries, sorts behind every
// barcode.  Per fragment id f < n: its barcode slot (a read of another barcode raises GF_FRAG_UMI), its read count and its
// smallest BAM index.  Ids >= n are ORed into frag_or (refused at the round trip) and left out of the tables.
#define UMI_EMPTY 0xffffffffffffffffull
#define FRAG_NONE 0xffffffffu
__global__ void k_umi_slots(const uint64_t* __restrict__ umi, const uint32_t* __restrict__ frag, int64_t n, unsigned long long* __restrict__ table,
                            uint32_t mask, uint32_t* __restrict__ frag_slot, uint32_t* __restrict__ frag_cnt, uint32_t* __restrict__ frag_min,
                            uint32_t* __restrict__ frag_ids, unsigned long long* __restrict__ frag_or, uint32_t* __restrict__ gflags) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned long long u = umi[i];
    const uint32_t f = frag[i];
    uint32_t h = hash64to32(u) & mask;
    for (;; ++h) {
        if (h == mask) h = 0;
        unsigned long long cur = table[h];
        if (cur == UMI_EMPTY) cur = atomicCAS(&table[h], UMI_EMPTY, u);
        if (cur == UMI_EMPTY || cur == u) break;
    }
    frag_ids[i] = (uint32_t)i;                                        // the payload of the fragment sort: every id, in id order
    if (f >= (uint64_t)n) { atomicOr(frag_or, (unsigned long long)f); return; }
    const uint32_t had = atomicCAS(&frag_slot[f], FRAG_NONE, h);
    if (had != FRAG_NONE && had != h) atomicOr(gflags, GF_FRAG_UMI);
    atomicAdd(&frag_cnt[f], 1u);
    atomicMin(&frag_min[f], (uint32_t)i);
}
// Fragment ids in barcode-slot order (stable: frag_id order inside a barcode; the ids no read carries last).  A real fragment's
// rank is its position j in that list.  ONE single-pass scan (decoupled look-back, smc_sort.cuh) over the barcode head flags and
// the read counts at once (two 31-bit counts in one word) gives every fragment its first sorted read position and its barcode
// rank; it writes urank / frank of every sorted read position, the barcode of every barcode rank, and frag_start[f], with
// FRAG_MULTI set for fragments of three or more reads (k_place_reads).
#define FRAG_MULTI 0x80000000u
__global__ void __launch_bounds__(SCAN_THREADS)
k_frag_scan(const uint32_t* __restrict__ slot_sorted, const uint32_t* __restrict__ frag_sorted, int64_t n, const uint32_t* __restrict__ frag_cnt,
            const uint32_t* __restrict__ frag_min, const uint64_t* __restrict__ umi, uint32_t* __restrict__ urank, uint32_t* __restrict__ frank,
            uint64_t* __restrict__ umi_of_urank, uint32_t* __restrict__ frag_start, unsigned long long* desc, uint32_t* counter, uint32_t* n_umi_out) {
    __shared__ unsigned long long warp_tot[SCAN_THREADS / 32];
    __shared__ uint32_t s_tile;
    __shared__ unsigned long long s_prefix;
    if (threadIdx.x == 0) s_tile = atomicAdd(counter, 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const int64_t base = (int64_t)tile * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
    unsigned long long v[SCAN_ITEMS], tsum = 0;                        // (barcode head << 31) | reads; 0 for an id without reads
    uint32_t prev = (base > 0 && base <= n) ? slot_sorted[base - 1] : FRAG_NONE;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        v[i] = 0;
        if (base + i < n) {
            const uint32_t s = slot_sorted[base + i];
            if (s != FRAG_NONE) v[i] = ((s != prev ? 1ull : 0ull) << 31) | frag_cnt[frag_sorted[base + i]];
            prev = s;
        }
        tsum += v[i];
    }
    unsigned long long incl = tsum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        unsigned long long t = __shfl_up_sync(FULL_MASK, incl, d);
        if (lane_id() >= (uint32_t)d) incl += t;
    }
    const int w = threadIdx.x >> 5;
    if (lane_id() == 31) warp_tot[w] = incl;
    __syncthreads();
    unsigned long long woff = 0, blk = 0;
#pragma unroll
    for (int i = 0; i < SCAN_THREADS / 32; ++i) {
        unsigned long long t = warp_tot[i];
        if (i < w) woff += t;
        blk += t;
    }
    if (threadIdx.x < 32) {
        const unsigned long long prefix = lb_resolve(desc, tile, blk);
        if (threadIdx.x == 0) {
            s_prefix = prefix;
            if (tile == gridDim.x - 1) *n_umi_out = (uint32_t)((prefix + blk) >> 31);
        }
    }
    __syncthreads();
    unsigned long long run = s_prefix + woff + incl - tsum;            // exclusive counts before the thread's first fragment
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        if (v[i] == 0) continue;
        const uint32_t start = (uint32_t)(run & 0x7fffffffull), cnt = (uint32_t)(v[i] & 0x7fffffffull), j = (uint32_t)(base + i);
        run += v[i];
        const uint32_t ur = (uint32_t)(run >> 31) - 1u, f = frag_sorted[j];
        SMC_BOUNDS((int64_t)start + cnt <= n && (int64_t)ur < n && (int64_t)f < n);
        for (uint32_t k = start; k < start + cnt; ++k) { urank[k] = ur; frank[k] = j; }
        if (v[i] >> 31) umi_of_urank[ur] = umi[frag_min[f]];
        frag_start[f] = start | (cnt > 2 ? FRAG_MULTI : 0u);
    }
}
// Sorted position of every read (inv[i], k_read_prep runs in BAM order): its fragment's first position plus its rank among the
// fragment's reads in BAM order, which for a fragment of one or two reads is whether it is not the smallest BAM index.  The reads
// of larger fragments take the positions of their fragment's range in arrival order (multi_read) and join multi_list, for
// k_rank_multi to rank them.
__global__ void k_place_reads(const uint32_t* __restrict__ frag, int64_t n, const uint32_t* __restrict__ frag_min, uint32_t* __restrict__ frag_start,
                              uint32_t* __restrict__ inv, uint32_t* __restrict__ multi_read, uint32_t* __restrict__ multi_list, uint32_t* __restrict__ n_multi) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t f = frag[i];
    if (f >= (uint64_t)n) { inv[i] = (uint32_t)i; return; }          // refused at the round trip; until then any position in range
    const uint32_t s = frag_start[f];
    if (!(s & FRAG_MULTI)) {
        inv[i] = s + ((uint32_t)i != frag_min[f] ? 1u : 0u);
        SMC_BOUNDS((int64_t)inv[i] < n);
        return;
    }
    const uint32_t p = atomicAdd(&frag_start[f], 1u) & ~FRAG_MULTI;   // FRAG_MULTI stays set: start + reads <= n < 2^31
    const uint32_t k = atomicAdd(n_multi, 1u);
    SMC_BOUNDS((int64_t)p < n && (int64_t)k < n);
    multi_read[p] = (uint32_t)i;
    multi_list[k] = (uint32_t)i;
}
// Reads of fragments of three or more reads (none in most batches): rank among the fragment's reads by BAM index.
__global__ void k_rank_multi(const uint32_t* __restrict__ multi_list, const uint32_t* __restrict__ n_multi, const uint32_t* __restrict__ frag,
                             const uint32_t* __restrict__ frag_cnt, const uint32_t* __restrict__ frag_start, const uint32_t* __restrict__ multi_read,
                             uint32_t* __restrict__ inv) {
    const uint32_t m = *n_multi;
    for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < m; t += gridDim.x * blockDim.x) {
        const uint32_t i = multi_list[t], f = frag[i], cnt = frag_cnt[f];
        const uint32_t start = (frag_start[f] & ~FRAG_MULTI) - cnt;   // k_place_reads advanced it by cnt
        uint32_t r = 0;
        for (uint32_t k = start; k < start + cnt; ++k) r += multi_read[k] < i ? 1u : 0u;
        SMC_BOUNDS(r < cnt);
        inv[i] = start + r;
    }
}
// (read x 32-locus tile) events: the number of tiles each read covers is scanned (single pass, look-back) and the events are
// written in the same kernel -- the only "event" that is ever materialised: one 12-byte row per (read x tile).  Events beyond
// `cap` are not written; the total always is (the host grows the buffers and launches again).
__global__ void __launch_bounds__(SCAN_THREADS)
k_expand_scan(const ReadRec* __restrict__ recs, int64_t n, uint64_t* __restrict__ ev_key, uint32_t* __restrict__ ev_val, uint32_t cap,
              unsigned long long* desc, uint32_t* counter, uint32_t* total) {
    __shared__ uint32_t warp_tot[SCAN_THREADS / 32];
    __shared__ uint32_t s_tile, s_prefix;
    if (threadIdx.x == 0) s_tile = atomicAdd(counter, 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const int w = threadIdx.x >> 5;
    const uint32_t lane = lane_id();
    // a warp owns 256 consecutive reads as SCAN_ITEMS rows of 32: lanes hold consecutive reads, so that the event writes of a row
    // land next to each other
    const int64_t wbase = (int64_t)tile * SCAN_TILE + (int64_t)w * (32 * SCAN_ITEMS);
    uint32_t t0[SCAN_ITEMS], cnt[SCAN_ITEMS], off[SCAN_ITEMS], run = 0;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        const int64_t r = wbase + i * 32 + lane;
        t0[i] = 0; cnt[i] = 0;
        if (r < n) {
            const int32_t lo = recs[r].lo, hi = recs[r].hi;
            if (hi > lo) { t0[i] = (uint32_t)lo >> 5; cnt[i] = ((uint32_t)(hi - 1) >> 5) - t0[i] + 1u; }
        }
        uint32_t incl = cnt[i];
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            uint32_t t = __shfl_up_sync(FULL_MASK, incl, d);
            if (lane >= (uint32_t)d) incl += t;
        }
        off[i] = run + incl - cnt[i];                         // exclusive offset inside the warp's 256 reads
        run += __shfl_sync(FULL_MASK, incl, 31);
    }
    if (lane == 0) warp_tot[w] = run;
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
            if (tile == gridDim.x - 1) *total = prefix + blk;
        }
    }
    __syncthreads();
    const uint32_t base_o = s_prefix + woff;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        uint32_t o = base_o + off[i];
        const uint32_t sidx = (uint32_t)(wbase + i * 32 + lane);
        for (uint32_t t = 0; t < cnt[i]; ++t, ++o)
            if (o < cap) { ev_key[o] = t0[i] + t; ev_val[o] = sidx; }
    }
}
// first event of every tile in the tile-sorted event list, and the number of warp units of the tile
__global__ void k_tile_offsets(const uint64_t* ev_key, int64_t ne, uint32_t n_tiles, uint32_t chunk, uint32_t* tile_off, uint32_t* unit_cnt) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t > n_tiles) return;
    const uint32_t a = ne > 0 ? (uint32_t)lower_bound_u64(ev_key, ne, (uint64_t)t) : 0u;
    tile_off[t] = a;
    uint32_t nev = 0;
    if (t < n_tiles) nev = (ne > 0 ? (uint32_t)lower_bound_u64(ev_key, ne, (uint64_t)t + 1ull) : 0u) - a;
    unit_cnt[t] = (nev + chunk - 1) / chunk;
}
// Dynamic-allele rows, grouped by locus and ordered by key inside a locus: count per locus, scan, place, and a tiny
// insertion sort per locus (a locus has a handful of such alleles) -- 7 launches instead of a 6-pass radix sort of a few
// thousand keys that was pure launch latency.
__global__ void k_dyn_count(const unsigned long long* __restrict__ dkey, uint32_t cap, uint32_t* __restrict__ cnt) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= cap) return;
    unsigned long long k = dkey[i];
    if (k != DYN_EMPTY) atomicAdd(&cnt[(uint32_t)(k >> DYN_LOCUS_SHIFT)], 1u);
}
__global__ void k_dyn_place(const unsigned long long* __restrict__ dkey, uint32_t cap, const uint32_t* __restrict__ first,
                            uint32_t* __restrict__ cursor, uint64_t* __restrict__ lk, uint32_t* __restrict__ lv) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= cap) return;
    unsigned long long k = dkey[i];
    if (k == DYN_EMPTY) return;
    const uint32_t L = (uint32_t)(k >> DYN_LOCUS_SHIFT);
    const uint32_t o = first[L] + atomicAdd(&cursor[L], 1u);
    lk[o] = k; lv[o] = i;
}
__global__ void k_dyn_sort_local(const uint32_t* __restrict__ first, int64_t n_loci, uint64_t* __restrict__ lk, uint32_t* __restrict__ lv) {
    int64_t L = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (L >= n_loci) return;
    const uint32_t a = first[L], b = first[L + 1];
    for (uint32_t i = a + 1; i < b; ++i) {
        const uint64_t k = lk[i]; const uint32_t v = lv[i];
        uint32_t j = i;
        while (j > a && lk[j - 1] > k) { lk[j] = lk[j - 1]; lv[j] = lv[j - 1]; --j; }
        lk[j] = k; lv[j] = v;
    }
}
__global__ void k_dyn_gather(const uint64_t* lk, const uint32_t* lv, int64_t n, const int32_t* dcnt, const unsigned long long* dlimb,
                             const uint8_t* diskey, const uint32_t* drep_read, const int32_t* drep_qpos, const int32_t* dlen,
                             unsigned long long* s_key, int32_t* s_cnt, unsigned long long* s_limb, uint8_t* s_iskey,
                             uint32_t* s_rep_read, int32_t* s_rep_qpos, int32_t* s_len) {
    int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    uint32_t e = lv[j];
    s_key[j] = lk[j];
    for (int c = 0; c < SMC_NCNT; ++c) s_cnt[j * SMC_NCNT + c] = dcnt[(size_t)e * SMC_NCNT + c];
    s_cnt[j * SMC_NCNT + SMC_C_REV] = dcnt[(size_t)e * SMC_NCNT + SMC_C_ALLELE] - dcnt[(size_t)e * SMC_NCNT + SMC_C_FWD];
    for (int t = 0; t < 3; ++t) s_limb[j * 3 + t] = dlimb[(size_t)e * 3 + t];
    s_iskey[j] = diskey[e];
    s_rep_read[j] = drep_read[e]; s_rep_qpos[j] = drep_qpos[e]; s_len[j] = dlen[e];
}
__global__ void k_sum_cvg(const int32_t* cvg, int64_t n, unsigned long long* out) {
    unsigned long long s = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) s += (unsigned)cvg[i];
    for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(FULL_MASK, s, d);
    if ((threadIdx.x & 31) == 0 && s) atomicAdd(out, s);
}

static inline unsigned nblk(int64_t n, int t) { return (unsigned)((n + t - 1) / t); }
#define LAUNCH(kern, grid, block, smem, ...)                        \
    do {                                                            \
        if ((grid) > 0) {                                           \
            kern<<<(grid), (block), (smem), ctx->st>>>(__VA_ARGS__); \
            ++g_launches;                                           \
        }                                                           \
    } while (0)

// ------------------------------------------------------------------------------------------------------------
extern "C" int smc_version(void) { return SMC_ABI_VERSION; }

extern "C" const char* smc_last_error(smc_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

extern "C" int smc_ctx_create(int device, const smc_params* params, smc_ctx** out) {
    if (!params || !out) { g_create_error = "smc_ctx_create: null argument"; return SMC_E_ARG; }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        g_create_error = std::string("smc_ctx_create: no CUDA device (") + cudaGetErrorString(e) + "); libsmc_b200 has no CPU fallback";
        return SMC_E_CUDA;
    }
    if (device < 0 || device >= ndev) { g_create_error = "smc_ctx_create: bad device index"; return SMC_E_ARG; }
    smc_ctx* ctx = new (std::nothrow) smc_ctx();
    if (!ctx) { g_create_error = "smc_ctx_create: out of host memory"; return SMC_E_ARG; }
    ctx->device = device; ctx->prm = *params;
    if (const char* ev = getenv("SMC_CHUNK")) { long v = atol(ev); if (v >= 64 && v <= 1000000) ctx->chunk = (uint32_t)v; }   // tuning knob
    auto fail = [&](const char* what, cudaError_t ce) {
        g_create_error = std::string(what) + ": " + cudaGetErrorString(ce);
        delete ctx; return SMC_E_CUDA;
    };
    if ((e = cudaSetDevice(device)) != cudaSuccess) return fail("cudaSetDevice", e);
    if ((e = cudaStreamCreateWithFlags(&ctx->st, cudaStreamNonBlocking)) != cudaSuccess) return fail("cudaStreamCreate", e);
    if ((e = cudaDeviceGetAttribute(&ctx->n_sm, cudaDevAttrMultiProcessorCount, device)) != cudaSuccess) return fail("cudaDeviceGetAttribute", e);
    for (DevBuf* b : ctx->bufs) b->st = ctx->st;
    {   // keep freed scratch in the pool for the next batch / context of this process
        cudaMemPool_t pool;
        unsigned long long keep = ~0ull;
        if ((e = cudaDeviceGetDefaultMemPool(&pool, device)) != cudaSuccess) return fail("cudaDeviceGetDefaultMemPool", e);
        if ((e = cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep)) != cudaSuccess) return fail("cudaMemPoolSetAttribute", e);
    }
    for (auto& ev : ctx->ev) if ((e = cudaEventCreate(&ev)) != cudaSuccess) return fail("cudaEventCreate", e);
    if ((e = cudaStreamCreateWithFlags(&ctx->st_copy, cudaStreamNonBlocking)) != cudaSuccess) return fail("cudaStreamCreate", e);
    if ((e = cudaEventCreateWithFlags(&ctx->ev_link, cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", e);
    if ((e = cudaEventCreateWithFlags(&ctx->ev_tmp, cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", e);
    if ((e = cudaEventCreateWithFlags(&ctx->ev_tmp2, cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", e);
    for (auto& ev : ctx->ev_chunk) if ((e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", e);
    // host-computed tables (glibc pow, the same libm CPython calls): 10^(-bq/10) and the PCR prior
    std::vector<double> bq(256);
    for (int q = 0; q < 256; ++q) bq[q] = std::pow(10.0, -(double)q / 10.0);                          // smCounter.py:469
    const size_t per = (size_t)(PCR_NMAX + 1) * (PCR_NMAX + 2) / 2;
    std::vector<double> pcr(3 * per);
    for (int k = 4; k <= 6; ++k)
        for (int n = 0; n <= PCR_NMAX; ++n)
            for (int c = 0; c <= n; ++c) {
                double ratio = ((double)c + 0.5) / ((double)n + 0.5 * (double)k);                       // :80
                pcr[(size_t)(k - 4) * per + (size_t)n * (n + 1) / 2 + c] = std::pow(10.0, -6.0 * ratio); // :81
            }
    if ((e = ctx->d_bqtab.ensure(256 * 8)) != cudaSuccess) return fail("cudaMalloc", e);
    if ((e = ctx->d_pcrtab.ensure(pcr.size() * 8)) != cudaSuccess) return fail("cudaMalloc", e);
    cudaMemcpy(ctx->d_bqtab.p, bq.data(), 256 * 8, cudaMemcpyHostToDevice);
    cudaMemcpy(ctx->d_pcrtab.p, pcr.data(), pcr.size() * 8, cudaMemcpyHostToDevice);
    if ((e = cudaFuncSetAttribute(k_merge_t<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, KB_SMEM_BYTES)) != cudaSuccess)
        return fail("cudaFuncSetAttribute(k_merge)", e);
    if ((e = cudaFuncSetAttribute(k_merge_t<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, KB_SMEM_BYTES)) != cudaSuccess)
        return fail("cudaFuncSetAttribute(k_merge list)", e);
    if ((e = cudaFuncSetAttribute(k_gather_t<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, KA_SMEM_BYTES(false))) != cudaSuccess)
        return fail("cudaFuncSetAttribute(k_gather)", e);
    if ((e = cudaFuncSetAttribute(k_gather_t<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, KA_SMEM_BYTES(true))) != cudaSuccess)
        return fail("cudaFuncSetAttribute(k_gather list)", e);
    // both pileup kernels want the shared-memory side of the L1 / shared split (their global loads are streamed once)
    cudaFuncSetAttribute(k_gather_t<false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    cudaFuncSetAttribute(k_gather_t<true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    cudaFuncSetAttribute(k_merge_t<false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    cudaFuncSetAttribute(k_merge_t<true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if ((e = radix_sort_init()) != cudaSuccess) return fail("cudaFuncSetAttribute(k_radix_scatter)", e);
    if ((e = ctx->d_small.ensure(4096)) != cudaSuccess) return fail("cudaMalloc", e);
    *out = ctx;
    return SMC_OK;
}

extern "C" void smc_ctx_destroy(smc_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->st_copy) cudaStreamSynchronize(ctx->st_copy);
    cudaStreamSynchronize(ctx->st);
    for (DevBuf* b : ctx->bufs) b->release();
    cudaStreamSynchronize(ctx->st);
    for (auto& ev : ctx->ev) if (ev) cudaEventDestroy(ev);
    for (auto& ev : ctx->ev_chunk) if (ev) cudaEventDestroy(ev);
    if (ctx->ev_tmp) cudaEventDestroy(ctx->ev_tmp);
    if (ctx->ev_tmp2) cudaEventDestroy(ctx->ev_tmp2);
    if (ctx->ev_link) {
        std::lock_guard<std::mutex> lk(g_link_mu);
        if (ctx->device >= 0 && ctx->device < 64 && g_link_owner[ctx->device] == ctx) { g_link_owner[ctx->device] = nullptr; g_link_tail[ctx->device] = nullptr; }
        cudaEventDestroy(ctx->ev_link);
    }
    if (ctx->st_copy) cudaStreamDestroy(ctx->st_copy);
    if (ctx->st) cudaStreamDestroy(ctx->st);
    free(ctx->h_bz_out);
    delete ctx;
}

// ------------------------------------------------------------------------------------------------------------
// Number of chunks the bases / qualities of a batch are uploaded in by smc_call_batch (1 = plain upload).
static int pipe_chunks_for(const smc_reads_soa* R) {
    if (const char* ev = getenv("SMC_PIPE_CHUNKS")) { long v = atol(ev); if (v >= 1 && v <= SMC_PIPE_MAX) return (int)v; }
    const int64_t payload = R->seq_bytes + R->qual_bytes;
    if (R->n_reads < 65536 || payload < (96ll << 20)) return 1;
    // A/B on B200, two contexts per GPU, 145 MB compact payload: 3 chunks 23.99 ms per 4 batches, 4: 24.11, 6: 24.49, 9: 24.51
    // (one context, 320 MB plain payload, round 1: 6 chunks 9.79 ms, 12: 9.57)
    const int64_t g = payload / (48ll << 20);
    return (int)(g < 2 ? 2 : g > 12 ? 12 : g);
}

static int qual_bits_of(const smc_reads_soa* R) { return (R->qual_bits == 4 || R->qual_bits == 2) ? R->qual_bits : 8; }
static int seq_bits_of(const smc_reads_soa* R) { return R->seq_bits == 2 ? 2 : 4; }
// words of bq[] a batch may need: a read stores (len + 1) / 2 bytes of 4-bit bases or (len + 3) / 4 bytes of 2-bit ones, and is
// padded to a multiple of four words
static int64_t bq_capacity(const smc_reads_soa* R) {
    return (seq_bits_of(R) == 4 ? 2 : 4) * R->seq_bytes + 4 * R->n_reads + 16;
}

// Every argument check of an upload.  It runs before anything is queued, so a rejected batch leaves the context as it was.
static int check_upload(const smc_reads_soa* R, const smc_loci* Lc, std::string& err) {
    if (!R || !Lc) { err = "smc_upload: null reads/loci"; return SMC_E_ARG; }
    if (R->n_reads < 0 || Lc->n_loci < 0) { err = "smc_upload: negative size"; return SMC_E_ARG; }
    if (Lc->n_loci > SMC_MAX_LOCI) { err = "smc_upload: more than 4194302 loci in one batch"; return SMC_E_LIMIT; }
    if (R->n_reads > (1ll << 30) || R->seq_bytes >= (1ll << 32) || R->qual_bytes >= (1ll << 32) || R->n_cigar_words >= (1ll << 32)) {
        err = "smc_upload: batch exceeds 2^30 reads or 4 GiB of bases/qualities/cigar; split the batch"; return SMC_E_LIMIT;
    }
    if (R->scalar_bits != 0 && R->scalar_bits != 32 && R->scalar_bits != 16 && R->scalar_bits != 8) { err = "smc_upload: scalar_bits must be 0, 8, 16 or 32"; return SMC_E_ARG; }
    if (R->qual_bits != 0 && R->qual_bits != 8 && R->qual_bits != 4 && R->qual_bits != 2) { err = "smc_upload: qual_bits must be 0, 2, 4 or 8"; return SMC_E_ARG; }
    if (qual_bits_of(R) != 8 && (R->qual_off || !R->qual_lut)) { err = "smc_upload: compact qualities need the packed layout (qual_off == NULL) and a qual_lut"; return SMC_E_ARG; }
    if (R->seq_bits != 0 && R->seq_bits != 4 && R->seq_bits != 2) { err = "smc_upload: seq_bits must be 0, 2 or 4"; return SMC_E_ARG; }
    if (seq_bits_of(R) == 2 && (R->seq_off || R->n_seq_exc < 0 || (R->n_seq_exc > 0 && (!R->seq_exc_read || !R->seq_exc_pos || !R->seq_exc_nib)))) {
        err = "smc_upload: compact bases need the packed layout (seq_off == NULL) and consistent exception arrays"; return SMC_E_ARG;
    }
    if ((R->ref_id_bits != 0 && R->ref_id_bits != 32 && R->ref_id_bits != 8) || (R->umi_bits != 0 && R->umi_bits != 64 && R->umi_bits != 32)) {
        err = "smc_upload: ref_id_bits must be 0, 8 or 32 and umi_bits 0, 32 or 64"; return SMC_E_ARG;
    }
    if ((R->store_lo == nullptr) != (R->store_len == nullptr)) { err = "smc_upload: store_lo and store_len must be given together"; return SMC_E_ARG; }
    if (bq_capacity(R) >= (1ll << 32)) {
        err = "smc_upload: the expanded bases / qualities of the batch exceed 4 GiB; split the batch"; return SMC_E_LIMIT;
    }
    return SMC_OK;
}

// Host -> device copies of one upload.  A chunked upload queues them on the copy stream while the compute stream runs the
// upload's kernels: a copy must not write a buffer the compute stream (re)allocated before the copy stream has waited for
// it, and a kernel must not read what the compute stream has not waited for (hand_over).
struct Upload {
    smc_ctx* ctx;
    bool split;                 // copies go to ctx->st_copy (else to ctx->st, in order with the kernels)
    bool grew = false;          // a buffer was (re)allocated on ctx->st since the copy stream last waited for it
    int64_t bytes = 0;          // bytes copied (smc_timings::bytes_h2d)
    cudaError_t ensure(DevBuf& b, size_t n) {
        if (n <= b.cap) return cudaSuccess;
        grew = true;
        return b.ensure(n);
    }
    cudaError_t copy(void* dst, const void* src, size_t n) {
        if (n == 0) return cudaSuccess;
        if (split && grew) {
            cudaError_t e = cudaEventRecord(ctx->ev_tmp, ctx->st);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->st_copy, ctx->ev_tmp, 0);
            if (e != cudaSuccess) return e;
            grew = false;
        }
        bytes += (int64_t)n;
        return cudaMemcpyAsync(dst, src, n, cudaMemcpyHostToDevice, split ? ctx->st_copy : ctx->st);
    }
    // a whole array, into a buffer grown to hold it (16 bytes at least, so that an empty array has an address too)
    cudaError_t copy(DevBuf& b, const void* src, size_t n) {
        const cudaError_t e = ensure(b, n ? n : 16);
        return e != cudaSuccess ? e : copy(b.p, src, n);
    }
    cudaError_t hand_over() {
        if (!split) return cudaSuccess;
        const cudaError_t e = cudaEventRecord(ctx->ev_tmp2, ctx->st_copy);
        return e != cudaSuccess ? e : cudaStreamWaitEvent(ctx->st, ctx->ev_tmp2, 0);
    }
};

// one k_widen launch: 8- / 16-bit values -> int32, 32-bit values -> int64
static void widen(smc_ctx* ctx, const void* in, int in_bytes, int64_t n, void* out) {
    if (in_bytes == 1) { auto k = k_widen<uint8_t, int32_t>; LAUNCH(k, nblk(n, 256), 256, 0, (const uint8_t*)in, n, (int32_t*)out); }
    else if (in_bytes == 2) { auto k = k_widen<uint16_t, int32_t>; LAUNCH(k, nblk(n, 256), 256, 0, (const uint16_t*)in, n, (int32_t*)out); }
    else { auto k = k_widen<uint32_t, int64_t>; LAUNCH(k, nblk(n, 256), 256, 0, (const uint32_t*)in, n, (int64_t*)out); }
}

// Offsets of a payload packed in read order: per-read sizes of k_pack_len `kind` scanned in place in `out`; their total goes to
// d_small word SW_PACK_TOTALS + total_word (smc_run_resident compares it with the payload size the caller declared).
static int pack_offsets(smc_ctx* ctx, int64_t n, int kind, int qbits, uint32_t* out, int total_word) {
    CK(ctx->d_scan.ensure((size_t)scan_scratch_words(n + 1) * 4 + 1024));
    LAUNCH(k_pack_len, nblk(n, 256), 256, 0, ctx->d_lseq.as<int32_t>(), ctx->has_store ? ctx->d_store_len.as<int32_t>() : nullptr,
           ctx->d_ncig.as<uint16_t>(), n, kind, qbits, out);
    exclusive_scan_u32(out, out, n, ctx->d_scan.as<uint32_t>(), ctx->d_small.as<uint32_t>() + SW_PACK_TOTALS + total_word, ctx->st);
    return SMC_OK;
}

// k_unpack grid (grid-stride over the reads): 8 blocks of 256 threads on each of the 148 SMs of a B200
static constexpr unsigned UNPACK_GRID = 148u * 8u;

// Uploaded bases / qualities -> bq[], for the reads expanded with upload chunk c (k_chunk_need; a one-chunk upload: all reads).
static void expand_payload(smc_ctx* ctx, int c, unsigned grid) {
    const int G = ctx->pipe_n > 1 ? ctx->pipe_n : 1;
    const uint32_t* first = G > 1 ? ctx->d_small.as<uint32_t>() + SW_CHUNK_FIRST : nullptr;
    const int64_t n = ctx->n_reads;
    const int32_t* store_len = ctx->has_store ? ctx->d_store_len.as<int32_t>() : nullptr;
    const bool b2 = ctx->seq_bits == 2;
    auto unpack = ctx->qual_bits == 2 ? (b2 ? k_unpack<2, 2> : k_unpack<2, 4>) : ctx->qual_bits == 4 ? (b2 ? k_unpack<4, 2> : k_unpack<4, 4>)
                                      : (b2 ? k_unpack<8, 2> : k_unpack<8, 4>);
    LAUNCH(unpack, grid, 256, 0, first, c, G, n, ctx->d_seq_poff.as<uint32_t>(), ctx->d_qual_poff.as<uint32_t>(), ctx->d_bq_off.as<uint32_t>(),
           ctx->bq_cap, ctx->d_lseq.as<int32_t>(), store_len, ctx->d_qual_lut.as<uint8_t>(), ctx->d_seq_up.as<uint8_t>(),
           ctx->d_qual_up.as<uint8_t>(), ctx->d_bq.as<uint16_t>());
    if (b2)                             // the bases of 2-bit uploads that are not A / C / G / T
        LAUNCH(k_patch_seq, nblk(ctx->n_seq_exc, 256), 256, 0, first, c, G, n, ctx->n_seq_exc, ctx->d_exc_read.as<uint32_t>(),
               ctx->d_exc_pos.as<uint32_t>(), ctx->d_exc_nib.as<uint8_t>(), ctx->d_bq_off.as<uint32_t>(), ctx->bq_cap, ctx->d_bq.as<uint16_t>());
}

// pipelined = false: everything on ctx->st, synchronised on return (smc_upload).
// pipelined = true : scalars / CIGAR / loci on ctx->st; bases and qualities in ctx->pipe_n chunks of equal byte size on
//                    ctx->st_copy, one event per chunk; returns without waiting (smc_call_batch synchronises both streams).
static int queue_upload(smc_ctx* ctx, const smc_reads_soa* R, const smc_loci* Lc, const smc_umi_keep* K, bool pipelined) {
    CK(cudaSetDevice(ctx->device));
    ctx->uploaded = false; ctx->ran = false;
    const int64_t n = R->n_reads, nl = Lc->n_loci;
    const size_t nz = (size_t)(n ? n : 1);
    const int G = pipelined ? pipe_chunks_for(R) : 1;
    ctx->pipe_n = 0;
    // A chunked batch sends EVERYTHING over the copy stream, in the order the kernels need it (scalars, CIGARs, loci, then
    // the chunks of bases / qualities): no copy waits for a kernel, so the link stays busy however long this context's --
    // or another context's -- kernels queue on the GPU.  The compute stream waits for what it consumes (hand_over).
    Upload up{ctx, pipelined && G > 1};
    static const bool link_turns = [] { const char* ev = getenv("SMC_LINK_TURNS"); return !(ev && atoi(ev) == 0); }();
    std::unique_lock<std::mutex> link_lock(g_link_mu, std::defer_lock);
    const int dv = ctx->device;
    if (up.split && link_turns && dv >= 0 && dv < 64) {
        link_lock.lock();
        if (g_link_tail[dv] && g_link_owner[dv] != ctx) CK(cudaStreamWaitEvent(ctx->st_copy, g_link_tail[dv], 0));
    }
    CK(cudaEventRecord(ctx->ev[EV_COPY_BEGIN], up.split ? ctx->st_copy : ctx->st));
    // per-read scalars; narrow ones (8- / 16-bit scalars, 8-bit reference indices, 32-bit barcode codes) are staged as they
    // are, 16-byte aligned, and widened on the device
    struct Narrow { const void* src; int bytes; DevBuf* dst; size_t stage_off; };
    Narrow narrow[6];
    int n_narrow = 0;
    size_t stage_bytes = 0;
    auto scalars = [&](DevBuf& dst, const void* src, int bytes, int wide_bytes) {
        if (bytes == wide_bytes) return up.copy(dst, src, (size_t)n * bytes);
        narrow[n_narrow++] = {src, bytes, &dst, stage_bytes};
        stage_bytes += ((size_t)n * bytes + 15) & ~(size_t)15;
        return dst.ensure(nz * (bytes == 4 ? 8 : 4));
    };
    const int sw = R->scalar_bits == 8 ? 1 : R->scalar_bits == 16 ? 2 : 4;      // bytes per nm / l_seq / store_lo / store_len
    CK(scalars(ctx->d_ref_id, R->ref_id, R->ref_id_bits == 8 ? 1 : 4, 4));
    CK(up.copy(ctx->d_pos, R->pos, (size_t)n * 4)); CK(up.copy(ctx->d_flag, R->flag, (size_t)n * 2));
    CK(up.copy(ctx->d_mapq, R->mapq, (size_t)n)); CK(up.copy(ctx->d_ncig, R->n_cigar, (size_t)n * 2));
    CK(up.copy(ctx->d_frag, R->frag_id, (size_t)n * 4));
    CK(scalars(ctx->d_umi, R->umi, R->umi_bits == 32 ? 4 : 8, 8));
    ctx->has_store = R->store_lo != nullptr;
    CK(scalars(ctx->d_nm, R->nm, sw, 4)); CK(scalars(ctx->d_lseq, R->l_seq, sw, 4));
    if (ctx->has_store) { CK(scalars(ctx->d_store_lo, R->store_lo, sw, 4)); CK(scalars(ctx->d_store_len, R->store_len, sw, 4)); }
    if (n_narrow) CK(up.ensure(ctx->d_stage, stage_bytes));
    for (int k = 0; k < n_narrow; ++k) CK(up.copy(ctx->d_stage.as<uint8_t>() + narrow[k].stage_off, narrow[k].src, (size_t)n * narrow[k].bytes));
    CK(up.hand_over());                     // the widening and the offsets below read the scalars
    for (int k = 0; k < n_narrow; ++k) widen(ctx, ctx->d_stage.as<uint8_t>() + narrow[k].stage_off, narrow[k].bytes, n, narrow[k].dst->p);
    const int qbits = qual_bits_of(R), sbits = seq_bits_of(R);
    ctx->qual_bits = qbits; ctx->seq_bits = sbits; ctx->n_seq_exc = sbits == 2 ? R->n_seq_exc : 0;
    // offsets: uploaded, or -- NULL = payload packed in read order -- computed here from l_seq / n_cigar (saves 24 B per read of
    // PCIe).  Bases and qualities: 32-bit byte offsets into the uploaded arrays (the caller's 64-bit ones are narrowed below).
    ctx->packed_seq = !R->seq_off; ctx->packed_qual = !R->qual_off; ctx->packed_cigar = !R->cigar_off;
    CK(ctx->d_seq_poff.ensure(nz * 4)); CK(ctx->d_qual_poff.ensure(nz * 4));
    if (R->seq_off) CK(up.copy(ctx->d_seq_off, R->seq_off, (size_t)n * 8));
    else if (const int rc = pack_offsets(ctx, n, sbits == 2 ? 4 : 0, 8, ctx->d_seq_poff.as<uint32_t>(), sbits == 2 ? 4 : 0)) return rc;
    if (R->qual_off) CK(up.copy(ctx->d_qual_off, R->qual_off, (size_t)n * 8));
    else if (const int rc = pack_offsets(ctx, n, qbits == 8 ? 1 : 3, qbits, ctx->d_qual_poff.as<uint32_t>(), qbits == 8 ? 1 : 3)) return rc;
    if (R->cigar_off) CK(up.copy(ctx->d_cig_off, R->cigar_off, (size_t)n * 8));
    else {
        CK(ctx->d_cig_off.ensure(nz * 8)); CK(ctx->d_v0.ensure(nz * 4));
        if (const int rc = pack_offsets(ctx, n, 2, 8, ctx->d_v0.as<uint32_t>(), 2)) return rc;
        widen(ctx, ctx->d_v0.p, 4, n, ctx->d_cig_off.p);
    }
    // the device layout: every read on a multiple of four bq[] words
    ctx->bq_cap = (uint32_t)bq_capacity(R);
    CK(ctx->d_bq_off.ensure(nz * 4)); CK(ctx->d_bq.ensure((size_t)ctx->bq_cap * 2));
    if (const int rc = pack_offsets(ctx, n, 5, 8, ctx->d_bq_off.as<uint32_t>(), 5)) return rc;
    if (qbits != 8) {
        CK(ctx->d_qual_lut.ensure(16));
        CK(cudaMemcpyAsync(ctx->d_qual_lut.p, R->qual_lut, qbits == 4 ? 16 : 4, cudaMemcpyHostToDevice, ctx->st));
    }
    if (sbits == 2) {          // the exceptions of the compact bases
        CK(up.copy(ctx->d_exc_read, R->seq_exc_read, (size_t)R->n_seq_exc * 4)); CK(up.copy(ctx->d_exc_pos, R->seq_exc_pos, (size_t)R->n_seq_exc * 4));
        CK(up.copy(ctx->d_exc_nib, R->seq_exc_nib, (size_t)R->n_seq_exc));
    }
    if (G == 1) { CK(up.copy(ctx->d_seq_up, R->seq, (size_t)R->seq_bytes)); CK(up.copy(ctx->d_qual_up, R->qual, (size_t)R->qual_bytes)); }
    CK(up.copy(ctx->d_cigar, R->cigar, (size_t)R->n_cigar_words * 4));
    CK(up.copy(ctx->d_loci_ref, Lc->ref_id, (size_t)nl * 4)); CK(up.copy(ctx->d_loci_pos, Lc->pos0, (size_t)nl * 4));
    CK(up.copy(ctx->d_loci_base, Lc->ref_base, (size_t)nl));
    ctx->has_keep = K && K->n_loci > 0;
    ctx->keep_n = ctx->has_keep ? K->n_loci : 0;
    ctx->keep_total = ctx->has_keep ? K->off[K->n_loci] : 0;
    ctx->ds_first_drawn = INT32_MAX;
    if (ctx->has_keep) {
        CK(up.copy(ctx->d_keep_off, K->off, (size_t)(K->n_loci + 1) * 8));
        CK(up.copy(ctx->d_keep_umi, K->umi, (size_t)K->off[K->n_loci] * 8));
        CK(up.copy(ctx->d_k0, K->locus, (size_t)K->n_loci * 8));              // d_k0 doubles as the staging buffer of the masked-locus list
    }
    CK(up.hand_over());
    {
        auto narrow = k_widen<int64_t, uint32_t>;
        if (R->seq_off) LAUNCH(narrow, nblk(n, 256), 256, 0, ctx->d_seq_off.as<int64_t>(), n, ctx->d_seq_poff.as<uint32_t>());
        if (R->qual_off) LAUNCH(narrow, nblk(n, 256), 256, 0, ctx->d_qual_off.as<int64_t>(), n, ctx->d_qual_poff.as<uint32_t>());
    }
    ctx->n_reads = n; ctx->n_loci = nl;
    if (G == 1) expand_payload(ctx, 0, std::min<unsigned>(nblk(n, 256) + 1u, UNPACK_GRID));
    if (ctx->has_keep) {
        CK(ctx->d_keep_idx.ensure((size_t)(nl ? nl : 1) * 4));
        LAUNCH(k_fill_i32, nblk(nl, 256), 256, 0, ctx->d_keep_idx.as<int32_t>(), nl, -1);
        LAUNCH(k_scatter_idx, nblk(K->n_loci, 256), 256, 0, ctx->d_k0.as<int64_t>(), K->n_loci, ctx->d_keep_idx.as<int32_t>());
    }
    CK(ctx->d_loci_key.ensure((size_t)(nl ? nl : 1) * 8));
    LAUNCH(k_loci_keys, nblk(nl, 256), 256, 0, ctx->d_loci_ref.as<int32_t>(), ctx->d_loci_pos.as<int32_t>(), nl, ctx->d_loci_key.as<uint64_t>());
    ctx->seq_bytes = R->seq_bytes; ctx->qual_bytes = R->qual_bytes; ctx->n_cigar_words = R->n_cigar_words;
    ctx->tm = smc_timings{};
    ctx->tm.n_reads = n; ctx->tm.n_loci = nl;
    if (G == 1) {
        CK(cudaEventRecord(ctx->ev[EV_COPY_END], ctx->st));
        if (!pipelined) {
            CK(cudaStreamSynchronize(ctx->st));
            cudaEventElapsedTime(&ctx->tm.ms_h2d, ctx->ev[EV_COPY_BEGIN], ctx->ev[EV_COPY_END]);
        }
    } else {
        // the chunks follow the scalars on the link; everything up to the first pileup launch needs the scalars only
        CK(up.ensure(ctx->d_seq_up, (size_t)R->seq_bytes + 16)); CK(up.ensure(ctx->d_qual_up, (size_t)R->qual_bytes + 16));
        auto chunk_bytes = [&](int64_t total) { int64_t c = (total + G - 1) / G; c = (c + 255) & ~255ll; return (uint32_t)std::max<int64_t>(c, 256); };
        const uint32_t seq_chunk = chunk_bytes(R->seq_bytes), qual_chunk = chunk_bytes(R->qual_bytes);
        // which reads each chunk lets k_unpack expand (k_read_prep turns it into the chunk every read's units wait for)
        uint32_t none[SMC_PIPE_MAX];
        for (int c = 0; c < SMC_PIPE_MAX; ++c) none[c] = (uint32_t)n;
        CK(cudaMemcpyAsync(ctx->d_small.as<uint32_t>() + SW_CHUNK_FIRST, none, sizeof(none), cudaMemcpyHostToDevice, ctx->st));
        LAUNCH(k_chunk_need, nblk(n, 256), 256, 0, ctx->d_seq_poff.as<uint32_t>(), ctx->d_qual_poff.as<uint32_t>(), ctx->d_lseq.as<int32_t>(),
               ctx->has_store ? ctx->d_store_len.as<int32_t>() : nullptr, n, sbits, qbits, seq_chunk, qual_chunk, G,
               ctx->d_small.as<uint32_t>() + SW_CHUNK_FIRST);
        for (int c = 0; c < G; ++c) {
            const int64_t s0 = std::min<int64_t>(R->seq_bytes, (int64_t)c * seq_chunk), s1 = std::min<int64_t>(R->seq_bytes, (int64_t)(c + 1) * seq_chunk);
            const int64_t q0 = std::min<int64_t>(R->qual_bytes, (int64_t)c * qual_chunk), q1 = std::min<int64_t>(R->qual_bytes, (int64_t)(c + 1) * qual_chunk);
            CK(up.copy(ctx->d_seq_up.as<uint8_t>() + s0, R->seq + s0, (size_t)(s1 - s0)));
            CK(up.copy(ctx->d_qual_up.as<uint8_t>() + q0, R->qual + q0, (size_t)(q1 - q0)));
            CK(cudaEventRecord(ctx->ev_chunk[c], ctx->st_copy));
        }
        CK(cudaEventRecord(ctx->ev[EV_COPY_END], ctx->st_copy));
        if (link_lock.owns_lock()) {
            CK(cudaEventRecord(ctx->ev_link, ctx->st_copy));
            g_link_tail[dv] = ctx->ev_link; g_link_owner[dv] = ctx;
        }
        ctx->pipe_n = G;
    }
    ctx->tm.pipe_chunks = pipelined ? G : 0;
    ctx->tm.bytes_h2d = up.bytes;
    ctx->uploaded = true;
    return SMC_OK;
}

static int upload_impl(smc_ctx* ctx, const smc_reads_soa* R, const smc_loci* Lc, const smc_umi_keep* K, bool pipelined) {
    if (!ctx) return SMC_E_ARG;
    NvtxRange nvtx_r("smc:upload");
    if (const int rc = check_upload(R, Lc, ctx->err)) return rc;
    const int rc = queue_upload(ctx, R, Lc, K, pipelined);
    if (rc != SMC_OK) {                     // no copy may still read the caller's buffers when an error is returned
        cudaStreamSynchronize(ctx->st_copy);
        cudaStreamSynchronize(ctx->st);
    }
    return rc;
}

extern "C" int smc_upload(smc_ctx* ctx, const smc_reads_soa* R, const smc_loci* Lc, const smc_umi_keep* K) {
    return upload_impl(ctx, R, Lc, K, false);
}

// One host round trip: `bytes` of device memory into `dst`, behind everything queued on ctx->st.
static int read_back(smc_ctx* ctx, void* dst, const void* src, size_t bytes) {
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->st));
    CK(cudaStreamSynchronize(ctx->st));
    return SMC_OK;
}

// K2a: order reads by (barcode, frag_id, BAM index).  Fragment ids are already in order inside a barcode and reads in BAM order
// inside a fragment, so it is the fragment ids that are sorted, stably on barcode slot; one single-pass scan over them gives the
// dense barcode / fragment ranks, the barcode of every rank and every fragment's first sorted position, from which each read
// takes its own (*inv: read index -> sorted position).  The two key buffers and the two payload buffers ping-pong in the sort;
// of the pair the sort does not leave its result in, the key buffer takes frag_start and the payload buffer inv, and once the
// scan has read the sorted pair, it takes the rare path's multi_read / multi_list.
static int read_sort(smc_ctx* ctx, const uint32_t** inv) {
    const int64_t n = ctx->n_reads;
    const size_t n4 = (size_t)n * 4;
    uint32_t* small = ctx->d_small.as<uint32_t>();
    CK(ctx->d_k0.ensure(n4)); CK(ctx->d_k1.ensure(n4)); CK(ctx->d_v0.ensure(n4)); CK(ctx->d_v1.ensure(n4));
    CK(ctx->d_frag_cnt.ensure(n4)); CK(ctx->d_frag_min.ensure(n4));
    CK(ctx->d_hist.ensure(radix_hist_words(n) * 4 + 1024));
    CK(ctx->d_scan.ensure((size_t)std::max<int64_t>(radix_scan_words(n), scan_scratch_words(n + 1)) * 4 + 1024));
    uint32_t* k0 = ctx->d_k0.as<uint32_t>(); uint32_t* k1 = ctx->d_k1.as<uint32_t>();
    uint32_t* v0 = ctx->d_v0.as<uint32_t>(); uint32_t* v1 = ctx->d_v1.as<uint32_t>();
    uint32_t* frag_cnt = ctx->d_frag_cnt.as<uint32_t>(); uint32_t* frag_min = ctx->d_frag_min.as<uint32_t>();
    // barcode table of >= 1.1 n slots (a batch has far fewer distinct barcodes than reads): a 2.9 M read panel batch sorts its
    // fragment ids on 22 key bits = two 11-bit passes
    int slot_bits = 4;
    while ((double)(1ll << slot_bits) < 1.1 * (double)n) ++slot_bits;
    CK(ctx->d_umi_table.ensure(((size_t)1 << slot_bits) * 8));
    CK(cudaMemsetAsync(ctx->d_umi_table.p, 0xff, ((size_t)1 << slot_bits) * 8, ctx->st));
    CK(cudaMemsetAsync(k0, 0xff, n4, ctx->st));                       // frag_slot = FRAG_NONE
    CK(cudaMemsetAsync(frag_min, 0xff, n4, ctx->st));
    CK(cudaMemsetAsync(frag_cnt, 0, n4, ctx->st));
    CK(cudaMemsetAsync(small + SW_FRAG_OR, 0, 8, ctx->st));
    CK(cudaMemsetAsync(small + SW_N_TILE_EVENTS, 0, 32, ctx->st));    // words 4 .. 11: tile-event total, gflags, ..., SW_N_MULTI
    LAUNCH(k_umi_slots, nblk(n, 256), 256, 0, ctx->d_umi.as<uint64_t>(), ctx->d_frag.as<uint32_t>(), n,
           ctx->d_umi_table.as<unsigned long long>(), (uint32_t)((1u << slot_bits) - 1u), k0, frag_cnt, frag_min, v0,
           (unsigned long long*)(small + SW_FRAG_OR), small + SW_GFLAGS);
    CK(cudaEventRecord(ctx->ev[EV_READ_SORT_BEGIN], ctx->st));
    const int res = radix_sort_bits(k0, v0, k1, v1, n, 0, slot_bits, ctx->d_hist.as<uint32_t>(), ctx->d_scan.as<uint32_t>(), ctx->st);
    CK(cudaEventRecord(ctx->ev[EV_READ_SORT_DONE], ctx->st));
    ctx->tm.read_sort_passes = n > 1 ? (slot_bits + RS_MAX_BITS - 1) / RS_MAX_BITS : 0;
    uint32_t* slot_sorted = res ? k1 : k0; uint32_t* frag_sorted = res ? v1 : v0;
    uint32_t* frag_start = res ? k0 : k1; uint32_t* inv_out = res ? v0 : v1;
    CK(ctx->d_urank.ensure(n4)); CK(ctx->d_frank.ensure(n4));
    CK(ctx->d_umi_of_urank.ensure((size_t)n * 8));
    const int64_t nbt = (n + SCAN_TILE - 1) / SCAN_TILE;
    uint32_t* scr = ctx->d_scan.as<uint32_t>();
    CK(cudaMemsetAsync(scr, 0, (size_t)(2 * nbt + 8) * 4, ctx->st));
    LAUNCH(k_frag_scan, (unsigned)nbt, SCAN_THREADS, 0, slot_sorted, frag_sorted, n, frag_cnt, frag_min, ctx->d_umi.as<uint64_t>(),
           ctx->d_urank.as<uint32_t>(), ctx->d_frank.as<uint32_t>(), ctx->d_umi_of_urank.as<uint64_t>(), frag_start,
           reinterpret_cast<unsigned long long*>(scr + 2), scr, small + SW_N_UMI);
    LAUNCH(k_place_reads, nblk(n, 256), 256, 0, ctx->d_frag.as<uint32_t>(), n, frag_min, frag_start, inv_out, slot_sorted, frag_sorted,
           small + SW_N_MULTI);
    LAUNCH(k_rank_multi, std::min<unsigned>(nblk(n, 256), 148u), 256, 0, frag_sorted, small + SW_N_MULTI, ctx->d_frag.as<uint32_t>(),
           frag_cnt, frag_start, slot_sorted, inv_out);
    *inv = inv_out;
    return SMC_OK;
}

// K1: per-read records, computed in BAM order (coalesced inputs) and stored at their sorted position
static int read_prep(smc_ctx* ctx, const uint32_t* inv) {
    const int64_t n = ctx->n_reads;
    uint32_t* small = ctx->d_small.as<uint32_t>();
    CK(ctx->d_recs.ensure((size_t)n * sizeof(ReadRec))); CK(ctx->d_grec.ensure((size_t)n * sizeof(GRec)));
    PrepArgs P{};
    P.n_reads = n; P.inv = inv; P.urank = ctx->d_urank.as<uint32_t>(); P.frank = ctx->d_frank.as<uint32_t>();
    P.ref_id = ctx->d_ref_id.as<int32_t>(); P.pos = ctx->d_pos.as<int32_t>(); P.flag = ctx->d_flag.as<uint16_t>();
    P.mapq = ctx->d_mapq.as<uint8_t>(); P.nm = ctx->d_nm.as<int32_t>(); P.l_seq = ctx->d_lseq.as<int32_t>();
    P.bq_off = ctx->d_bq_off.as<uint32_t>(); P.cigar_off = ctx->d_cig_off.as<int64_t>();
    P.n_cigar = ctx->d_ncig.as<uint16_t>(); P.cigar = ctx->d_cigar.as<uint32_t>();
    if (ctx->has_store) { P.store_lo = ctx->d_store_lo.as<int32_t>(); P.store_len = ctx->d_store_len.as<int32_t>(); }
    P.loci_key = ctx->d_loci_key.as<uint64_t>(); P.n_loci = ctx->n_loci;
    P.minMQ = ctx->prm.minMQ; P.primerDist = ctx->prm.primerDist; P.mismatchThr = ctx->prm.mismatchThr;
    P.recs = ctx->d_recs.as<ReadRec>(); P.grec = ctx->d_grec.as<GRec>(); P.gflags = small + SW_GFLAGS;
    if (ctx->pipe_n > 1) {
        CK(ctx->d_pipe_need.ensure((size_t)n));
        P.pipe_need = ctx->d_pipe_need.as<uint8_t>(); P.pipe_n = (uint32_t)ctx->pipe_n; P.chunk_first = small + SW_CHUNK_FIRST;
    }
    CK(cudaEventRecord(ctx->ev[EV_READ_PREP_BEGIN], ctx->st));
    LAUNCH(k_read_prep, nblk(n, 256), 256, 0, P);
    CK(cudaEventRecord(ctx->ev[EV_READ_PREP_DONE], ctx->st));
    ctx->tm.read_prep_bytes = n * (int64_t)(4 + 4 + 2 + 1 + 4 + 4 + 4 + 8 + 2 + (ctx->has_store ? 8 : 0) + 4 + sizeof(ReadRec) + sizeof(GRec)) + 4 * ctx->n_cigar_words;
    return SMC_OK;
}

// The input checks only the device can make, from d_small words 0 .. SW_PACK_TOTALS + 5 as the read sort, k_read_prep and the
// upload left them (w[i] = word i).
static int check_device_inputs(smc_ctx* ctx, const uint32_t* w) {
    const uint32_t gflags = w[SW_GFLAGS];
    if (gflags & GF_BAD_READ) { ctx->err = "a read has l_seq or clip length > 65535 (unsupported)"; return SMC_E_LIMIT; }
    if (gflags & GF_BAD_STORE) {
        ctx->err = "stored window: store_lo must be even and >= 0, store_lo + store_len <= l_seq, reads with indels / clips inside must be "
                   "stored whole, and every target base of a read must lie inside its window";
        return SMC_E_ARG;
    }
    if (w[SW_FRAG_OR] | w[SW_FRAG_OR + 1]) { ctx->err = "frag_id must be a dense id (< n_reads), numbered by first appearance"; return SMC_E_ARG; }
    if (gflags & GF_FRAG_UMI) { ctx->err = "a frag_id must belong to one barcode"; return SMC_E_ARG; }
    const uint32_t* tot = w + SW_PACK_TOTALS;
    if ((ctx->packed_seq && (int64_t)tot[ctx->seq_bits == 2 ? 4 : 0] != ctx->seq_bytes) || (ctx->packed_qual && (int64_t)tot[ctx->qual_bits != 8 ? 3 : 1] != ctx->qual_bytes) ||
        (ctx->packed_cigar && (int64_t)tot[2] != ctx->n_cigar_words)) {
        ctx->err = "packed payload (NULL offsets): seq_bytes / qual_bytes / n_cigar_words do not match the sums of (len+1)/2, len, n_cigar (len = store_len or l_seq)";
        return SMC_E_ARG;
    }
    if (tot[5] > ctx->bq_cap) {             // only a caller's offsets can get here: the packed sizes bound the words
        ctx->err = "the reads' bases (l_seq or store_len) need more room than seq_bytes provides";
        return SMC_E_ARG;
    }
    return SMC_OK;
}

// k_expand_scan into event buffers of ctx->ne_cap entries: events beyond them are not written, their total always is
static int expand_tile_events(smc_ctx* ctx) {
    const int64_t n = ctx->n_reads;
    if (ctx->ne_cap > 0xfffffff0ll) ctx->ne_cap = 0xfffffff0ll;
    CK(ctx->d_ek0.ensure((size_t)ctx->ne_cap * 8)); CK(ctx->d_ev0.ensure((size_t)ctx->ne_cap * 4));
    const int64_t nbt = (n + SCAN_TILE - 1) / SCAN_TILE;
    uint32_t* scr = ctx->d_scan.as<uint32_t>();
    CK(cudaMemsetAsync(scr, 0, (size_t)(2 * nbt + 8) * 4, ctx->st));
    LAUNCH(k_expand_scan, (unsigned)nbt, SCAN_THREADS, 0, ctx->d_recs.as<ReadRec>(), n, ctx->d_ek0.as<uint64_t>(), ctx->d_ev0.as<uint32_t>(),
           (uint32_t)ctx->ne_cap, reinterpret_cast<unsigned long long*>(scr + 2), scr, ctx->d_small.as<uint32_t>() + SW_N_TILE_EVENTS);
    return SMC_OK;
}

// K2b (first half): the (read x tile) events, written into buffers sized from the previous batch (or 4 per read).  The round
// trip after them brings back their exact count, the barcode count and the device-side input checks; the first batch of a
// shape whose events did not fit grows the buffers and writes them again.
static int tile_events(smc_ctx* ctx) {
    if (ctx->ne_cap < 4 * ctx->n_reads + 4096) ctx->ne_cap = 4 * ctx->n_reads + 4096;
    if (const int rc = expand_tile_events(ctx)) return rc;
    uint32_t w[SW_PACK_TOTALS + 6];
    if (const int rc = read_back(ctx, w, ctx->d_small.p, sizeof(w))) return rc;
    if (const int rc = check_device_inputs(ctx, w)) return rc;
    ctx->tm.n_umi_groups = w[SW_N_UMI];
    ctx->n_tile_events = w[SW_N_TILE_EVENTS];
    if (ctx->n_tile_events <= ctx->ne_cap) return SMC_OK;
    ctx->ne_cap = ctx->n_tile_events + ctx->n_tile_events / 8 + 4096;
    return expand_tile_events(ctx);
}

// K2b: the events, stable sort by tile; first event and warp units of every tile; [eb, ee) of every unit, cut at barcode
// boundaries
static int sort_tiles(smc_ctx* ctx) {
    const int64_t NE = ctx->n_tile_events;
    const uint32_t n_tiles = (uint32_t)((ctx->n_loci + 31) / 32);
    CK(cudaEventRecord(ctx->ev[EV_EVENT_SORT_BEGIN], ctx->st));
    const uint64_t* ev_key_sorted = nullptr;
    ctx->ev_read_sorted = nullptr;
    CK(ctx->d_tile_off.ensure((size_t)(n_tiles + 2) * 4)); CK(ctx->d_unit_cnt.ensure((size_t)(n_tiles + 2) * 4));
    CK(ctx->d_unit_off.ensure((size_t)(n_tiles + 2) * 4));
    if (NE > 0) {
        CK(ctx->d_ek1.ensure((size_t)NE * 8)); CK(ctx->d_ev1.ensure((size_t)NE * 4));
        CK(ctx->d_hist.ensure(radix_hist_words(NE) * 4 + 1024));
        CK(ctx->d_scan.ensure((size_t)std::max<int64_t>(radix_scan_words(NE), scan_scratch_words((int64_t)n_tiles + 2)) * 4 + 1024));
        int tile_bits = 0;                                             // a panel batch of <= 2048 tiles is ONE pass
        while (((uint64_t)(n_tiles - 1) >> tile_bits) != 0) ++tile_bits;
        int res = radix_sort_bits(ctx->d_ek0.as<uint64_t>(), ctx->d_ev0.as<uint32_t>(), ctx->d_ek1.as<uint64_t>(), ctx->d_ev1.as<uint32_t>(),
                                  NE, 0, tile_bits, ctx->d_hist.as<uint32_t>(), ctx->d_scan.as<uint32_t>(), ctx->st);
        ev_key_sorted = res ? ctx->d_ek1.as<uint64_t>() : ctx->d_ek0.as<uint64_t>();
        ctx->ev_read_sorted = res ? ctx->d_ev1.as<uint32_t>() : ctx->d_ev0.as<uint32_t>();
    } else {
        CK(ctx->d_scan.ensure((size_t)scan_scratch_words((int64_t)n_tiles + 2) * 4 + 1024));
    }
    CK(cudaEventRecord(ctx->ev[EV_EVENT_SORT_DONE], ctx->st));
    LAUNCH(k_tile_offsets, nblk((int64_t)n_tiles + 1, 256), 256, 0, ev_key_sorted, NE, n_tiles, ctx->chunk, ctx->d_tile_off.as<uint32_t>(),
           ctx->d_unit_cnt.as<uint32_t>());
    exclusive_scan_u32(ctx->d_unit_cnt.as<uint32_t>(), ctx->d_unit_off.as<uint32_t>(), (int64_t)n_tiles + 1, ctx->d_scan.as<uint32_t>(),
                       nullptr, ctx->st);
    const int64_t max_units = (int64_t)n_tiles + NE / ctx->chunk + 1;
    ctx->n_units_cap = (uint32_t)max_units;
    CK(ctx->d_unit_eb.ensure((size_t)max_units * 4)); CK(ctx->d_unit_ee.ensure((size_t)max_units * 4));
    CK(ctx->d_unit_tile.ensure((size_t)max_units * 4)); CK(ctx->d_unit_nfrag.ensure((size_t)max_units * 4));
    LAUNCH(k_unit_bounds, nblk(max_units, 256), 256, 0, ctx->d_tile_off.as<uint32_t>(), ctx->d_unit_off.as<uint32_t>(), n_tiles, ctx->chunk,
           ctx->ev_read_sorted, ctx->d_urank.as<uint32_t>(), ctx->d_unit_eb.as<uint32_t>(), ctx->d_unit_ee.as<uint32_t>(),
           ctx->d_unit_tile.as<uint32_t>(), ctx->n_units_cap);
    return SMC_OK;
}

// Chunked upload: which units may start after which chunk.  A unit needs the latest chunk any of its reads needs (k_read_prep:
// pipe_need); pipe_end[c] is the end of the units that chunks 0 .. c complete.
static int plan_chunks(smc_ctx* ctx) {
    const int G = ctx->pipe_n;
    uint32_t init[SMC_PIPE_MAX], blocked[SMC_PIPE_MAX];
    for (int c = 0; c < SMC_PIPE_MAX; ++c) init[c] = ctx->n_units_cap;
    uint32_t* pd = ctx->d_small.as<uint32_t>() + SW_PIPE_BLOCKED;
    CK(cudaMemcpyAsync(pd, init, sizeof(init), cudaMemcpyHostToDevice, ctx->st));
    LAUNCH(k_pipe_unit_need, nblk((int64_t)ctx->n_units_cap * 32, 256), 256, 0, ctx->d_unit_eb.as<uint32_t>(),
           ctx->d_unit_ee.as<uint32_t>(), ctx->ev_read_sorted, ctx->d_pipe_need.as<uint8_t>(), ctx->n_units_cap, pd);
    if (const int rc = read_back(ctx, blocked, pd, sizeof(blocked))) return rc;
    uint32_t run = ctx->n_units_cap;
    for (int c = G - 1; c >= 0; --c) {
        if (c < G - 1) run = std::min(run, blocked[c]);
        ctx->pipe_end[c] = run;
    }
    return SMC_OK;
}

static DynTab make_dyntab(smc_ctx* ctx) {
    uint32_t* small = ctx->d_small.as<uint32_t>();
    DynTab T;
    T.dkey = ctx->d_dkey.as<unsigned long long>(); T.dmask = ctx->dyn_cap - 1; T.drep_read = ctx->d_drep_read.as<uint32_t>();
    T.drep_qpos = ctx->d_drep_qpos.as<int32_t>(); T.dlen = ctx->d_dlen.as<int32_t>(); T.dcnt = ctx->d_dcnt.as<int32_t>();
    T.dlimb = ctx->d_dlimb.as<unsigned long long>(); T.diskey = ctx->d_diskey.as<uint8_t>(); T.dcount = small + SW_DYN_COUNT; T.gflags = small + SW_GFLAGS;
    T.bq = ctx->d_bq.as<uint16_t>(); T.bq_off = ctx->d_bq_off.as<uint32_t>();
    return T;
}

// Scratch of the K3a -> K3b hand-over: fragment codes (+ first-read indices when listing, + barcode ranks when a mask or a
// listing needs the barcode of a closing run).
static int ensure_code_storage(smc_ctx* ctx, bool list, bool need_uranks) {
    const uint64_t slots = code_slots_total((uint64_t)ctx->n_tile_events, ctx->n_units_cap, ctx->code_mult);
    CK(ctx->d_codes.ensure((size_t)slots * 64));
    if (list) CK(ctx->d_frag_first.ensure((size_t)slots * 128));
    if (need_uranks) CK(ctx->d_umi_urank.ensure((size_t)(ctx->n_tile_events + 1) * 4));
    return SMC_OK;
}

static void fill_kargs(smc_ctx* ctx, KAArgs& A, KBArgs& B, bool list, bool need_uranks) {
    A = KAArgs{}; B = KBArgs{};
    A.grec = ctx->d_grec.as<GRec>(); A.recs = ctx->d_recs.as<ReadRec>(); A.ev_read = ctx->ev_read_sorted;
    A.urank_s = ctx->d_urank.as<uint32_t>(); A.frank_s = ctx->d_frank.as<uint32_t>();
    A.unit_eb = ctx->d_unit_eb.as<uint32_t>(); A.unit_ee = ctx->d_unit_ee.as<uint32_t>(); A.unit_tile = ctx->d_unit_tile.as<uint32_t>();
    A.n_units = ctx->n_units_cap; A.code_mult = ctx->code_mult;
    A.loci_pos = ctx->d_loci_pos.as<int32_t>(); A.n_loci = ctx->n_loci;
    A.bq = ctx->d_bq.as<uint16_t>(); A.cigar = ctx->d_cigar.as<uint32_t>();
    A.minBQ = ctx->prm.minBQ; A.primerDist = ctx->prm.primerDist;
    A.codes = ctx->d_codes.as<uint4>(); A.unit_nfrag = ctx->d_unit_nfrag.as<uint32_t>();
    A.frag_first = list ? ctx->d_frag_first.as<uint32_t>() : nullptr;
    A.umi_urank = need_uranks ? ctx->d_umi_urank.as<uint32_t>() : nullptr;
    A.loc = ctx->d_loc.as<int32_t>(); A.cnt = ctx->d_cnt.as<int32_t>();
    A.T = make_dyntab(ctx);

    B.codes = ctx->d_codes.as<uint4>(); B.unit_nfrag = ctx->d_unit_nfrag.as<uint32_t>(); B.frag_first = A.frag_first; B.umi_urank = A.umi_urank;
    B.unit_eb = A.unit_eb; B.unit_ee = A.unit_ee; B.unit_tile = A.unit_tile; B.n_units = A.n_units; B.code_mult = A.code_mult;
    B.n_loci = ctx->n_loci;
    B.bqtab = ctx->d_bqtab.as<double>(); B.pcrtab = ctx->d_pcrtab.as<double>(); B.pcr_nmax = PCR_NMAX;
    B.mtDrop = ctx->prm.mtDrop;
    B.smt = ctx->prm.rpb < 1.5 ? 2.0 : ctx->prm.rpb < 3.0 ? 3.0 : 4.0;                     // smCounter.py:303-308
    B.keep_idx = ctx->has_keep ? ctx->d_keep_idx.as<int32_t>() : nullptr;
    B.keep_off = ctx->d_keep_off.as<int64_t>(); B.keep_umi = ctx->d_keep_umi.as<uint64_t>();
    B.umi_of_urank = ctx->d_umi_of_urank.as<uint64_t>();
    B.loc = ctx->d_loc.as<int32_t>(); B.cnt = ctx->d_cnt.as<int32_t>(); B.limb = ctx->d_limb.as<unsigned long long>();
    B.T = A.T;
    B.list_idx = nullptr;
    B.defer = ctx->d_defer.as<uint4>(); B.defer_cap = ctx->defer_cap; B.defer_count = ctx->d_small.as<uint32_t>() + SW_DEFER_COUNT;
}

// k_gather + k_merge over units [0, n_units_cap): one pair, or for a chunked upload one pair per range [pipe_end[c-1],
// pipe_end[c]) that starts once chunk c is in (after expanding its reads' bases and qualities when `expand`); then
// k_merge_deferred over the barcodes the k_merge launches deferred (the list's count is cleared by the caller).
// `gather_done`, unless null, is recorded between the kernels of the one pair, or after the last pair of a chunked run.
template <bool LIST>
static int launch_pileup(smc_ctx* ctx, KAArgs& A, KBArgs& B, bool chunked, bool expand, cudaEvent_t gather_done) {
    if (chunked) ctx->tm.pipe_launches = 0;
    uint32_t u0 = 0;
    for (int c = 0; c < (chunked ? ctx->pipe_n : 1); ++c) {
        if (chunked) {
            CK(cudaStreamWaitEvent(ctx->st, ctx->ev_chunk[c], 0));
            if (expand) expand_payload(ctx, c, UNPACK_GRID);
        }
        const uint32_t u1 = chunked ? ctx->pipe_end[c] : ctx->n_units_cap;
        if (u1 <= u0) continue;
        A.unit0 = B.unit0 = u0; A.n_units = B.n_units = u1;
        LAUNCH(k_gather_t<LIST>, nblk(u1 - u0, KA_WARPS), KA_WARPS * 32, KA_SMEM_BYTES(LIST), A);
        if (gather_done && !chunked) CK(cudaEventRecord(gather_done, ctx->st));
        LAUNCH(k_merge_t<LIST>, nblk(u1 - u0, KB_WARPS), KB_WARPS * 32, KB_SMEM_BYTES, B);
        u0 = u1;
        if (chunked) ++ctx->tm.pipe_launches;
    }
    if (gather_done && chunked) CK(cudaEventRecord(gather_done, ctx->st));
    // the record count is only known on the device: at most one wave of threads, each walks the list with a grid stride
    LAUNCH(k_merge_deferred, std::min<unsigned>(nblk(ctx->defer_cap, KD_THREADS), 148u * 8u), KD_THREADS, 0, B);
    return SMC_OK;
}

// Initial length of the deferred-barcode list of k_merge: one record per 32 tile events, never below 1024.  The batches of cfg2
// (6.9 - 10.4 M tile events) defer 14.7 k - 25.6 k (barcode, locus) pairs, about one per 400 tile events; a batch that
// defers more runs its pileup again with the list grown x4, and the context keeps the longer list.
static uint32_t defer_cap_for(int64_t n_tile_events) {
    return (uint32_t)std::min<int64_t>(std::max<int64_t>(1024, n_tile_events / 32), 1ll << 24);
}

// K3: the pileup, into per-locus accumulators and a dynamic-allele table cleared for it.  The round trip after it brings back
// the overflow flags: a pileup that overflowed the dynamic-allele table, the fragment-code storage or the deferred-barcode list
// runs again with the one that overflowed grown.
static int pileup(smc_ctx* ctx) {
    NvtxRange nvtx_r("smc:pileup");
    const size_t nlz = (size_t)(ctx->n_loci ? ctx->n_loci : 1);
    uint32_t* small = ctx->d_small.as<uint32_t>();
    CK(ctx->d_loc.ensure(nlz * SMC_NLOC * 4)); CK(ctx->d_cnt.ensure(nlz * SMC_NFIXED * SMC_NCNT * 4));
    CK(ctx->d_limb.ensure(nlz * SMC_NFIXED * 3 * 8)); CK(ctx->d_pi.ensure(nlz * SMC_NFIXED * 8));
    CK(ctx->d_max.ensure(nlz * 4)); CK(ctx->d_second.ensure(nlz * 4)); CK(ctx->d_alt.ensure(nlz * 4));
    CK(ctx->d_altpi.ensure(nlz * 8)); CK(ctx->d_secondpi.ensure(nlz * 8)); CK(ctx->d_fl1.ensure(nlz * 4)); CK(ctx->d_fl2.ensure(nlz * 4));
    CK(ctx->d_bial.ensure(nlz)); CK(ctx->d_fp.ensure(nlz * 8 * 8)); CK(ctx->d_for.ensure(nlz * 8 * 8));
    CK(ctx->d_dyn_first.ensure((nlz + 2) * 4));
    if (ctx->dyn_cap == 0) {
        uint32_t want = 1u << 16;
        while ((int64_t)want < 2 * ctx->n_loci && want < (1u << 28)) want <<= 1;
        if (const char* ev = getenv("SMC_DYN_CAP0")) {            // test hook: start small to exercise the regrowth path
            long v = atol(ev);
            if (v >= 16 && v <= (1l << 28) && (v & (v - 1)) == 0) want = (uint32_t)v;
        }
        ctx->dyn_cap = want;
    }
    if (const char* ev = ctx->defer_cap == 0 ? getenv("SMC_SPILL_CAP0") : nullptr) {     // test hook: start small to exercise the regrowth path
        const long v = atol(ev);
        if (v >= 1 && v <= (1l << 24)) ctx->defer_cap = (uint32_t)v;
    } else {
        ctx->defer_cap = std::max(ctx->defer_cap, defer_cap_for(ctx->n_tile_events));
    }
    for (int attempt = 0;; ++attempt) {
        const uint32_t cap = ctx->dyn_cap;
        CK(ctx->d_dkey.ensure((size_t)cap * 8)); CK(ctx->d_drep_read.ensure((size_t)cap * 4)); CK(ctx->d_drep_qpos.ensure((size_t)cap * 4));
        CK(ctx->d_dlen.ensure((size_t)cap * 4)); CK(ctx->d_dcnt.ensure((size_t)cap * SMC_NCNT * 4)); CK(ctx->d_dlimb.ensure((size_t)cap * 24));
        CK(ctx->d_diskey.ensure(cap));
        CK(cudaMemsetAsync(ctx->d_dkey.p, 0xff, (size_t)cap * 8, ctx->st));
        CK(cudaMemsetAsync(ctx->d_drep_read.p, 0xff, (size_t)cap * 4, ctx->st));      // "not published yet" (dyn_lookup_long_ins)
        CK(cudaMemsetAsync(ctx->d_dcnt.p, 0, (size_t)cap * SMC_NCNT * 4, ctx->st));
        CK(cudaMemsetAsync(ctx->d_dlimb.p, 0, (size_t)cap * 24, ctx->st));
        CK(cudaMemsetAsync(ctx->d_diskey.p, 0, cap, ctx->st));
        CK(cudaMemsetAsync(ctx->d_loc.p, 0, nlz * SMC_NLOC * 4, ctx->st));
        CK(cudaMemsetAsync(ctx->d_cnt.p, 0, nlz * SMC_NFIXED * SMC_NCNT * 4, ctx->st));
        CK(cudaMemsetAsync(ctx->d_limb.p, 0, nlz * SMC_NFIXED * 3 * 8, ctx->st));
        CK(cudaMemsetAsync(small + SW_GFLAGS, 0, 24, ctx->st));     // gflags, dyn count, n_tasks, cvg sum
        CK(ctx->d_defer.ensure((size_t)ctx->defer_cap * sizeof(uint4)));
        CK(cudaMemsetAsync(small + SW_DEFER_COUNT, 0, 4, ctx->st));
        if (ctx->n_tile_events > 0) {
            if (const int rc = ensure_code_storage(ctx, false, ctx->has_keep)) return rc;
            KAArgs A; KBArgs B;
            fill_kargs(ctx, A, B, false, ctx->has_keep);
            CK(cudaEventRecord(ctx->ev[EV_PILEUP_BEGIN], ctx->st));
            if (const int rc = launch_pileup<false>(ctx, A, B, ctx->pipe_n > 1, attempt == 0, ctx->ev[EV_GATHER_DONE])) return rc;
            CK(cudaEventRecord(ctx->ev[EV_MERGE_DONE], ctx->st));
        }
        uint32_t w[2];                                               // d_small words SW_GFLAGS, SW_DYN_COUNT
        if (const int rc = read_back(ctx, w, small + SW_GFLAGS, sizeof(w))) return rc;
        CK(cudaGetLastError());
        const uint32_t gflags = w[0];
        if (!(gflags & (GF_DYN_FULL | GF_CODE_FULL | GF_DEFER_FULL))) { ctx->n_dyn = w[1]; return SMC_OK; }
        if (gflags & GF_DEFER_FULL) ctx->defer_cap = ctx->defer_cap >= (1u << 26) ? ctx->defer_cap : ctx->defer_cap * 4;
        if (attempt == 5) { ctx->err = "dynamic allele table / fragment code storage overflow"; return SMC_E_OVERFLOW; }
        if (gflags & GF_CODE_FULL) ctx->code_mult = 3;             // worst-case layout: always fits
        if (gflags & GF_DYN_FULL) {
            if (ctx->dyn_cap >= (1u << 28)) { ctx->err = "dynamic allele table overflow"; return SMC_E_OVERFLOW; }
            ctx->dyn_cap <<= 2;
        }
    }
}

// Dynamic alleles -> rows grouped by locus, ordered by key inside a locus
static int dyn_rows(smc_ctx* ctx) {
    NvtxRange nvtx_r("smc:dyn_rows");
    const int64_t nl = ctx->n_loci, nd = ctx->n_dyn;
    const size_t nlz = (size_t)(nl ? nl : 1), ndz = (size_t)(nd ? nd : 1);
    CK(ctx->d_s_key.ensure(ndz * 8)); CK(ctx->d_s_cnt.ensure(ndz * SMC_NCNT * 4)); CK(ctx->d_s_limb.ensure(ndz * 24));
    CK(ctx->d_s_iskey.ensure(ndz)); CK(ctx->d_s_pi.ensure(ndz * 8)); CK(ctx->d_s_rep_read.ensure(ndz * 4));
    CK(ctx->d_s_rep_qpos.ensure(ndz * 4)); CK(ctx->d_s_len.ensure(ndz * 4));
    CK(cudaMemsetAsync(ctx->d_dyn_first.p, 0, (nlz + 2) * 4, ctx->st));
    if (nd == 0) return SMC_OK;
    CK(ctx->d_lk0.ensure(ndz * 8)); CK(ctx->d_lv0.ensure(ndz * 4)); CK(ctx->d_lv1.ensure((nlz + 2) * 4));
    CK(ctx->d_scan.ensure((size_t)scan_scratch_words((int64_t)nl + 2) * 4 + 1024));
    uint32_t* first = ctx->d_dyn_first.as<uint32_t>();
    uint32_t* cursor = ctx->d_lv1.as<uint32_t>();
    CK(cudaMemsetAsync(cursor, 0, (nlz + 2) * 4, ctx->st));
    LAUNCH(k_dyn_count, nblk(ctx->dyn_cap, 256), 256, 0, ctx->d_dkey.as<unsigned long long>(), ctx->dyn_cap, first);
    exclusive_scan_u32(first, first, nl + 1, ctx->d_scan.as<uint32_t>(), nullptr, ctx->st);
    LAUNCH(k_dyn_place, nblk(ctx->dyn_cap, 256), 256, 0, ctx->d_dkey.as<unsigned long long>(), ctx->dyn_cap, first, cursor,
           ctx->d_lk0.as<uint64_t>(), ctx->d_lv0.as<uint32_t>());
    LAUNCH(k_dyn_sort_local, nblk(nl, 256), 256, 0, first, nl, ctx->d_lk0.as<uint64_t>(), ctx->d_lv0.as<uint32_t>());
    LAUNCH(k_dyn_gather, nblk(nd, 128), 128, 0, ctx->d_lk0.as<uint64_t>(), ctx->d_lv0.as<uint32_t>(), nd, ctx->d_dcnt.as<int32_t>(),
           ctx->d_dlimb.as<unsigned long long>(),
           ctx->d_diskey.as<uint8_t>(), ctx->d_drep_read.as<uint32_t>(), ctx->d_drep_qpos.as<int32_t>(), ctx->d_dlen.as<int32_t>(),
           ctx->d_s_key.as<unsigned long long>(), ctx->d_s_cnt.as<int32_t>(), ctx->d_s_limb.as<unsigned long long>(),
           ctx->d_s_iskey.as<uint8_t>(), ctx->d_s_rep_read.as<uint32_t>(), ctx->d_s_rep_qpos.as<int32_t>(), ctx->d_s_len.as<int32_t>());
    return SMC_OK;
}

// ds = maxMT or round(2 * mtDepth) (smCounter.py:486)
static int ds_of(const smc_ctx* ctx) {
    return ctx->prm.maxMT > 0 ? ctx->prm.maxMT : (int)std::llround(2.0 * (double)ctx->prm.mtDepth);
}

// K4: k_call (PI, ALT, filters, Fisher task list), k_fisher, and the sum of cvg.  The round trip after them brings back the task
// count: a list longer than its buffer is grown and the three kernels run once more.
static int call_stats(smc_ctx* ctx) {
    NvtxRange nvtx_r("smc:call+fisher");
    const int64_t nl = ctx->n_loci;
    uint32_t* small = ctx->d_small.as<uint32_t>();
    for (int attempt = 0;; ++attempt) {
        if (ctx->task_cap == 0) ctx->task_cap = 1u << 13;
        CK(ctx->d_tasks.ensure((size_t)ctx->task_cap * sizeof(FisherTask)));
        CK(cudaMemsetAsync(small + SW_N_TASKS, 0, 4, ctx->st));
        K4Args B{};
        B.n_loci = nl; B.ref_base = ctx->d_loci_base.as<uint8_t>(); B.loc = ctx->d_loc.as<int32_t>(); B.cnt = ctx->d_cnt.as<int32_t>();
        B.limb = ctx->d_limb.as<unsigned long long>(); B.pi = ctx->d_pi.as<double>();
        B.n_dyn = ctx->n_dyn; B.dyn_key = ctx->d_s_key.as<unsigned long long>(); B.dyn_cnt = ctx->d_s_cnt.as<int32_t>();
        B.dyn_limb = ctx->d_s_limb.as<unsigned long long>(); B.dyn_iskey = ctx->d_s_iskey.as<uint8_t>(); B.dyn_pi = ctx->d_s_pi.as<double>();
        B.dyn_first = ctx->d_dyn_first.as<uint32_t>();
        B.keep_idx = ctx->has_keep ? ctx->d_keep_idx.as<int32_t>() : nullptr;
        B.ds = ds_of(ctx);
        B.ds_first_drawn = ctx->ds_first_drawn;
        if (ctx->ds_mode == SMC_DS_DEVICE) {
            B.ds_count = small + SW_DS_LOCI;
            CK(cudaMemsetAsync(small + SW_DS_LOCI, 0, 12, ctx->st));
        }
        B.max_allele = ctx->d_max.as<int32_t>(); B.second_allele = ctx->d_second.as<int32_t>(); B.alt_allele = ctx->d_alt.as<int32_t>();
        B.alt_pi = ctx->d_altpi.as<double>(); B.second_pi = ctx->d_secondpi.as<double>(); B.fl1 = ctx->d_fl1.as<uint32_t>();
        B.fl2 = ctx->d_fl2.as<uint32_t>(); B.biallelic = ctx->d_bial.as<uint8_t>(); B.fisher_p = ctx->d_fp.as<double>();
        B.fisher_or = ctx->d_for.as<double>(); B.tasks = ctx->d_tasks.as<FisherTask>(); B.n_tasks = small + SW_N_TASKS; B.task_cap = ctx->task_cap;
        LAUNCH(k_call, nblk(nl, 128), 128, 0, B);
        // k_fisher reads the task count on the device: launched for the whole task buffer (idle threads leave at once), so
        // that no host round trip sits between the two kernels; an overflowing task list is noticed at the round trip below
        LAUNCH(k_fisher, nblk((int64_t)ctx->task_cap * 32, 128), 128, 0, ctx->d_tasks.as<FisherTask>(), small + SW_N_TASKS, ctx->task_cap, nl, (int)ctx->prm.fisherLegacy,
               ctx->d_fp.as<double>(), ctx->d_for.as<double>(), ctx->d_fl1.as<uint32_t>(), ctx->d_fl2.as<uint32_t>());
        CK(cudaMemsetAsync(small + SW_CVG_SUM, 0, 8, ctx->st));
        LAUNCH(k_sum_cvg, std::min<unsigned>(nblk(nl, 256), 592u), 256, 0, ctx->d_loc.as<int32_t>() + (size_t)SMC_L_CVG * nl, nl,
               (unsigned long long*)(small + SW_CVG_SUM));
        CK(cudaEventRecord(ctx->ev[EV_STATS_DONE], ctx->st));
        uint32_t w[9];                                               // d_small words SW_N_TASKS, SW_CVG_SUM (u64), .. SW_DS_LOCI, SW_DS_LOCI + 1 (u64)
        const size_t nw = ctx->ds_mode == SMC_DS_DEVICE ? 9 : 3;
        if (const int rc = read_back(ctx, w, small + SW_N_TASKS, nw * 4)) return rc;
        CK(cudaGetLastError());
        const uint32_t n_tasks = w[0];
        if (n_tasks <= ctx->task_cap) {
            ctx->tm.n_fisher = n_tasks;
            ctx->tm.n_pileup_events = (int64_t)(w[1] | (uint64_t)w[2] << 32);
            ctx->ds_flagged = nw == 9 ? w[SW_DS_LOCI - SW_N_TASKS] : 0;
            ctx->ds_barcodes = nw == 9 ? (int64_t)(w[SW_DS_LOCI + 1 - SW_N_TASKS] | (uint64_t)w[SW_DS_LOCI + 2 - SW_N_TASKS] << 32) : 0;
            return SMC_OK;
        }
        if (attempt == 1) { ctx->err = "Fisher task list overflow"; return SMC_E_OVERFLOW; }
        ctx->task_cap = n_tasks + n_tasks / 4 + 1024;                // grow and redo the (cheap) call kernel
    }
}

// ------------------------------------------------------------------------------------------------------------
// Down-sampling drawn on the device (smc_downsample.cuh)

// draw scratch of one k_ds_draw launch: sets beyond it go to further launches (a set alone may exceed it)
static constexpr int64_t DS_WAVE_WORDS = 1ll << 30;

static int bit_length(uint64_t v) { return v ? 64 - __builtin_clzll(v) : 0; }

// k_ds_draw over the sets [0, nsets) of the device offsets d_off (total keys), in waves whose scratch stays within
// DS_WAVE_WORDS; host_off are the same offsets on the host, or null (then read back when one wave does not hold them all)
static int draw_sets(smc_ctx* ctx, const int64_t* d_off, const int64_t* host_off, int64_t nsets, int64_t total, const int64_t* d_pos1,
                     const int32_t* d_locus, const int64_t* d_k, int64_t ds, const int64_t* d_hash, uint32_t* d_out) {
    auto at = [](const int64_t* off, int64_t k) { return 16 * (off[k] + k) + (PY2_MT_N + 16) * k; };
    const int64_t all = 16 * (total + nsets) + (PY2_MT_N + 16) * nsets;
    std::vector<int64_t> off_h;
    if (all > DS_WAVE_WORDS && !host_off) {
        off_h.resize((size_t)nsets + 1);
        if (const int rc = read_back(ctx, off_h.data(), d_off, off_h.size() * 8)) return rc;
        host_off = off_h.data();
    }
    for (int64_t k0 = 0; k0 < nsets;) {
        int64_t k1 = nsets, words = all;
        if (all > DS_WAVE_WORDS) {
            k1 = k0 + 1;
            while (k1 < nsets && at(host_off, k1 + 1) - at(host_off, k0) <= DS_WAVE_WORDS) ++k1;
            words = at(host_off, k1) - at(host_off, k0);
        }
        CK(ctx->d_ds_scratch.ensure((size_t)words * 4));
        LAUNCH(k_ds_draw, nblk(k1 - k0, 64), 64, 0, d_off, k0, k1, d_pos1, d_locus, ctx->d_loci_pos.as<int32_t>(), d_k, ds, d_hash,
               ctx->d_ds_scratch.as<uint32_t>(), d_out);
        k0 = k1;
    }
    return SMC_OK;
}

// k_ds_hash over `total` codes; fails with SMC_E_ARG naming a dictionary-coded barcode without a hash.  *code_or: OR of the codes.
static int hash_barcodes(smc_ctx* ctx, const uint32_t* order, const uint64_t* umi, int64_t total, uint64_t* code_or) {
    uint32_t* small = ctx->d_small.as<uint32_t>();
    CK(ctx->d_ds_codes.ensure((size_t)total * 8)); CK(ctx->d_ds_hash.ensure((size_t)total * 8));
    CK(cudaMemsetAsync(small + SW_DS_MISSING, 0, 16, ctx->st));
    LAUNCH(k_ds_hash, nblk(total, 256), 256, 0, order, umi, total, ctx->d_bc_code.as<uint64_t>(), ctx->d_bc_hash.as<int64_t>(), ctx->n_bc,
           ctx->d_ds_codes.as<uint64_t>(), ctx->d_ds_hash.as<int64_t>(), (unsigned long long*)(small + SW_DS_MISSING),
           (unsigned long long*)(small + SW_DS_OR));
    uint64_t w[2];
    if (const int rc = read_back(ctx, w, small + SW_DS_MISSING, sizeof(w))) return rc;
    CK(cudaGetLastError());
    if (w[0]) {
        char code[24];
        snprintf(code, sizeof(code), "0x%016llx", (unsigned long long)w[0]);
        ctx->err = std::string("no Py2 hash for the dictionary-coded barcode ") + code + " (smc_set_barcode_hashes)";
        return SMC_E_ARG;
    }
    *code_or = w[1];
    return SMC_OK;
}

// The loci call_stats flagged SMC_ST_NEED_DOWNSAMPLE: number them and list their barcodes, order each locus's barcodes by first
// passing read, hash them, draw ds of them per locus, merge the kept codes (ascending per locus) into the mask CSR behind the
// caller's masks, and run the pileup and the statistics again on the resident batch.
static int device_downsample(smc_ctx* ctx) {
    NvtxRange nvtx_r("smc:downsample");
    const int64_t nl = ctx->n_loci, nflag = ctx->ds_flagged, T = ctx->ds_barcodes, ds = ds_of(ctx), m = nflag * ds;
    if (T > 0xffffffffll) { ctx->err = "down-sampling: more than 2^32 barcodes at the flagged loci of one batch; split the batch"; return SMC_E_LIMIT; }
    const size_t tz = (size_t)(T ? T : 1), wz = (size_t)std::max<int64_t>(std::max<int64_t>(nl, T), 1);
    CK(ctx->d_ds_flag.ensure((size_t)nl * 4)); CK(ctx->d_ds_nbc.ensure((size_t)nl * 4)); CK(ctx->d_list_idx.ensure((size_t)nl * 4));
    CK(ctx->d_list_off.ensure((size_t)(nflag + 1) * 8)); CK(ctx->d_ds_locus.ensure((size_t)nflag * 4)); CK(ctx->d_list_count.ensure((size_t)nflag * 4));
    CK(ctx->d_ds_v0.ensure(wz * 4)); CK(ctx->d_ds_v1.ensure(wz * 4)); CK(ctx->d_ds_k0.ensure(tz * 8)); CK(ctx->d_ds_k1.ensure(tz * 8));
    CK(ctx->d_list_umi.ensure(tz * 8)); CK(ctx->d_list_first.ensure(tz * 4));
    CK(ctx->d_hist.ensure(radix_hist_words(T) * 4 + 1024));
    CK(ctx->d_scan.ensure((size_t)std::max<int64_t>(radix_scan_words(T), scan_scratch_words(nl)) * 4 + 1024));
    uint32_t *v0 = ctx->d_ds_v0.as<uint32_t>(), *v1 = ctx->d_ds_v1.as<uint32_t>();
    uint64_t *k0 = ctx->d_ds_k0.as<uint64_t>(), *k1 = ctx->d_ds_k1.as<uint64_t>();
    int64_t* list_off = ctx->d_list_off.as<int64_t>();
    int32_t* locus = ctx->d_ds_locus.as<int32_t>();
    // 1. ordinal and first listed barcode of every flagged locus
    LAUNCH(k_ds_flags, nblk(nl, 256), 256, 0, ctx->d_loc.as<int32_t>(), nl, ctx->d_ds_flag.as<uint32_t>(), ctx->d_ds_nbc.as<uint32_t>());
    exclusive_scan_u32(ctx->d_ds_flag.as<uint32_t>(), v0, nl, ctx->d_scan.as<uint32_t>(), nullptr, ctx->st);
    exclusive_scan_u32(ctx->d_ds_nbc.as<uint32_t>(), v1, nl, ctx->d_scan.as<uint32_t>(), nullptr, ctx->st);
    LAUNCH(k_ds_list_fill, nblk(nl, 256), 256, 0, ctx->d_ds_flag.as<uint32_t>(), v0, v1, nl, nflag, T, ctx->d_list_idx.as<int32_t>(), list_off, locus);
    // 2. their barcodes with their first passing reads: the listing pass of the pileup pair
    CK(cudaMemsetAsync(ctx->d_list_count.p, 0, (size_t)nflag * 4, ctx->st));
    CK(cudaMemsetAsync(ctx->d_small.as<uint32_t>() + SW_DEFER_COUNT, 0, 4, ctx->st));
    if (const int rc = ensure_code_storage(ctx, true, true)) return rc;
    {
        KAArgs A; KBArgs B;
        fill_kargs(ctx, A, B, true, true);
        B.keep_idx = nullptr;
        B.list_idx = ctx->d_list_idx.as<int32_t>(); B.list_count = ctx->d_list_count.as<uint32_t>();
        B.list_off = list_off; B.list_umi = ctx->d_list_umi.as<uint64_t>(); B.list_first = ctx->d_list_first.as<uint32_t>(); B.list_cap = T;
        if (const int rc = launch_pileup<true>(ctx, A, B, false, false, nullptr)) return rc;
    }
    // 3. bcDict insertion order: (locus, first passing read); 4. the hashes in that order
    LAUNCH(k_ds_sort_keys, nblk(T, 256), 256, 0, list_off, nflag, ctx->d_list_first.as<uint32_t>(), T, k0, v0);
    const int r1 = radix_sort_bits(k0, v0, k1, v1, T, 0, 30 + bit_length((uint64_t)(nflag - 1)), ctx->d_hist.as<uint32_t>(), ctx->d_scan.as<uint32_t>(), ctx->st);
    uint64_t code_or = 0;
    if (const int rc = hash_barcodes(ctx, r1 ? v1 : v0, ctx->d_list_umi.as<uint64_t>(), T, &code_or)) return rc;
    // 5. the draw: insertion indices of the kept barcodes, ds per locus, then their codes in ascending order per locus
    if (const int rc = draw_sets(ctx, list_off, nullptr, nflag, T, nullptr, locus, nullptr, ds, ctx->d_ds_hash.as<int64_t>(), v0)) return rc;
    const uint32_t* order = nullptr;
    uint64_t* code_sorted = ctx->d_ds_codes.as<uint64_t>();
    if (m > 0) {
        LAUNCH(k_ds_kept, nblk(m, 256), 256, 0, list_off, m, ds, ctx->d_ds_codes.as<uint64_t>(), k0, v0);
        const int r2 = radix_sort_bits(k0, v0, k1, v1, m, 0, bit_length(code_or), ctx->d_hist.as<uint32_t>(), ctx->d_scan.as<uint32_t>(), ctx->st);
        uint64_t* ka = r2 ? k1 : k0; uint32_t* va = r2 ? v1 : v0;
        LAUNCH(k_ds_group_keys, nblk(m, 256), 256, 0, m, ds, ka, va, code_sorted);
        const int r3 = radix_sort_bits(ka, va, r2 ? k0 : k1, r2 ? v0 : v1, m, 0, bit_length((uint64_t)(nflag - 1)), ctx->d_hist.as<uint32_t>(),
                                       ctx->d_scan.as<uint32_t>(), ctx->st);
        order = r3 ? (r2 ? v0 : v1) : va;
    }
    // 6. the mask CSR: the caller's masks first, then the drawn ones
    const int64_t n_keep = ctx->keep_n + nflag, keep_total = ctx->keep_total + m;
    CK(ctx->d_ds_keep_off.ensure((size_t)(n_keep + 1) * 8)); CK(ctx->d_ds_keep_umi.ensure((size_t)std::max<int64_t>(keep_total, 1) * 8));
    if (ctx->keep_n > 0) {
        CK(cudaMemcpyAsync(ctx->d_ds_keep_off.p, ctx->d_keep_off.p, (size_t)ctx->keep_n * 8, cudaMemcpyDeviceToDevice, ctx->st));
        CK(cudaMemcpyAsync(ctx->d_ds_keep_umi.p, ctx->d_keep_umi.p, (size_t)ctx->keep_total * 8, cudaMemcpyDeviceToDevice, ctx->st));
    }
    if (!ctx->has_keep) {
        CK(ctx->d_keep_idx.ensure((size_t)nl * 4));
        LAUNCH(k_fill_i32, nblk(nl, 256), 256, 0, ctx->d_keep_idx.as<int32_t>(), nl, -1);
    }
    LAUNCH(k_ds_csr, nblk(std::max<int64_t>(nflag + 1, m), 256), 256, 0, nflag, ds, ctx->keep_n, ctx->keep_total, locus, order, code_sorted,
           ctx->d_keep_idx.as<int32_t>(), ctx->d_ds_keep_off.as<int64_t>(), ctx->d_ds_keep_umi.as<uint64_t>());
    std::swap(ctx->d_keep_off.p, ctx->d_ds_keep_off.p); std::swap(ctx->d_keep_off.cap, ctx->d_ds_keep_off.cap);
    std::swap(ctx->d_keep_umi.p, ctx->d_ds_keep_umi.p); std::swap(ctx->d_keep_umi.cap, ctx->d_ds_keep_umi.cap);
    ctx->has_keep = true;
    ctx->ds_first_drawn = (int32_t)ctx->keep_n;
    ctx->keep_n = n_keep; ctx->keep_total = keep_total;
    // 7. the batch again, every base and quality already expanded
    ctx->pipe_n = 0;
    if (const int rc = pileup(ctx)) return rc;
    if (const int rc = dyn_rows(ctx)) return rc;
    return call_stats(ctx);
}

// smc_timings of the run: the stage times from the events the stages that ran recorded, and the work counts
static void record_timings(smc_ctx* ctx) {
    smc_timings& t = ctx->tm;
    auto ms = [ctx](float* out, StageEvent from, StageEvent to) { cudaEventElapsedTime(out, ctx->ev[from], ctx->ev[to]); };
    ms(&t.ms_prep, EV_RUN_BEGIN, EV_PREP_DONE);
    ms(&t.ms_sort, EV_PREP_DONE, EV_SORT_DONE);
    ms(&t.ms_pileup, EV_SORT_DONE, EV_PILEUP_DONE);
    ms(&t.ms_stats, EV_PILEUP_DONE, EV_STATS_DONE);
    ms(&t.ms_total_device, EV_RUN_BEGIN, EV_STATS_DONE);
    ms(&t.ms_event_sort, EV_EVENT_SORT_BEGIN, EV_EVENT_SORT_DONE);
    t.ms_read_sort = t.ms_k_read_prep = 0.f;
    if (ctx->n_reads > 0 && ctx->n_loci > 0) {
        ms(&t.ms_read_sort, EV_READ_SORT_BEGIN, EV_READ_SORT_DONE);
        ms(&t.ms_k_read_prep, EV_READ_PREP_BEGIN, EV_READ_PREP_DONE);
    }
    t.ms_k_pileup = t.ms_k_gather = t.ms_k_merge = 0.f;
    if (ctx->n_tile_events > 0) {
        ms(&t.ms_k_pileup, EV_PILEUP_BEGIN, EV_MERGE_DONE);
        ms(&t.ms_k_gather, EV_PILEUP_BEGIN, EV_GATHER_DONE);
        ms(&t.ms_k_merge, EV_GATHER_DONE, EV_MERGE_DONE);
    }
    t.n_tile_events = ctx->n_tile_events;
    t.n_dyn = ctx->n_dyn;
    t.kernel_launches = g_launches;
    t.code_mult = (int32_t)ctx->code_mult; t.dyn_capacity = (int32_t)ctx->dyn_cap;
}

// One batch run of the resident upload, stage by stage.  Host round trips: after the tile events (their count and the
// device-side input checks), after the chunk plan (chunked uploads only), after the pileup and after the statistics; the
// tile events, the pileup and the statistics run once more when one of their buffers turned out too small.
extern "C" int smc_run_resident(smc_ctx* ctx) {
    if (!ctx) return SMC_E_ARG;
    if (!ctx->uploaded) { ctx->err = "smc_run_resident: nothing uploaded"; return SMC_E_STATE; }
    CK(cudaSetDevice(ctx->device));
    g_launches = 0;
    ctx->n_tile_events = 0;
    CK(cudaEventRecord(ctx->ev[EV_RUN_BEGIN], ctx->st));
    if (ctx->n_reads > 0 && ctx->n_loci > 0) {
        NvtxRange nvtx_r("smc:read_sort+prep+tile_events");
        const uint32_t* inv = nullptr;
        if (const int rc = read_sort(ctx, &inv)) return rc;
        if (const int rc = read_prep(ctx, inv)) return rc;
        if (const int rc = tile_events(ctx)) return rc;
    }
    CK(cudaEventRecord(ctx->ev[EV_PREP_DONE], ctx->st));
    if (const int rc = sort_tiles(ctx)) return rc;
    if (ctx->pipe_n > 1 && ctx->n_tile_events > 0)
        if (const int rc = plan_chunks(ctx)) return rc;
    CK(cudaEventRecord(ctx->ev[EV_SORT_DONE], ctx->st));
    if (const int rc = pileup(ctx)) return rc;
    CK(cudaEventRecord(ctx->ev[EV_PILEUP_DONE], ctx->st));
    if (const int rc = dyn_rows(ctx)) return rc;
    if (const int rc = call_stats(ctx)) return rc;
    if (ctx->ds_flagged > 0)
        if (const int rc = device_downsample(ctx)) return rc;
    record_timings(ctx);
    ctx->ran = true;
    return SMC_OK;
}

// Device -> host copies of one download; an output array the caller left NULL is skipped.
struct Download {
    smc_ctx* ctx;
    int64_t bytes = 0;          // bytes copied (smc_timings::bytes_d2h)
    template <class T> cudaError_t copy(T* dst, const DevBuf& src, size_t count) {
        if (!dst || count == 0) return cudaSuccess;
        bytes += (int64_t)(count * sizeof(T));
        return cudaMemcpyAsync(dst, src.p, count * sizeof(T), cudaMemcpyDeviceToHost, ctx->st);
    }
};

extern "C" int smc_download(smc_ctx* ctx, smc_out* out) {
    if (!ctx) return SMC_E_ARG;
    if (!ctx->ran) { ctx->err = "smc_download: nothing has been run"; return SMC_E_STATE; }
    if (!out || out->n_loci != ctx->n_loci) { ctx->err = "smc_download: smc_out.n_loci does not match the uploaded loci"; return SMC_E_ARG; }
    CK(cudaSetDevice(ctx->device));
    const size_t nl = (size_t)ctx->n_loci;
    const int64_t nd = ctx->n_dyn;
    out->n_dyn = nd;
    if (nd > out->dyn_capacity) { ctx->err = "smc_download: dyn_capacity too small (n_dyn reported in smc_out.n_dyn)"; return SMC_E_LIMIT; }
    NvtxRange nvtx_r("smc:download");
    Download down{ctx};
    CK(cudaEventRecord(ctx->ev[EV_COPY_BEGIN], ctx->st));
    CK(down.copy(out->loc, ctx->d_loc, nl * SMC_NLOC)); CK(down.copy(out->cnt, ctx->d_cnt, nl * SMC_NFIXED * SMC_NCNT));
    CK(down.copy(out->pi, ctx->d_pi, nl * SMC_NFIXED)); CK(down.copy(out->max_allele, ctx->d_max, nl));
    CK(down.copy(out->second_allele, ctx->d_second, nl)); CK(down.copy(out->alt_allele, ctx->d_alt, nl));
    CK(down.copy(out->alt_pi, ctx->d_altpi, nl)); CK(down.copy(out->second_pi, ctx->d_secondpi, nl));
    CK(down.copy(out->fl1, ctx->d_fl1, nl)); CK(down.copy(out->fl2, ctx->d_fl2, nl)); CK(down.copy(out->biallelic, ctx->d_bial, nl));
    CK(down.copy(out->fisher_p, ctx->d_fp, nl * 8)); CK(down.copy(out->fisher_or, ctx->d_for, nl * 8));
    CK(down.copy(out->dyn_cnt, ctx->d_s_cnt, (size_t)nd * SMC_NCNT)); CK(down.copy(out->dyn_pi, ctx->d_s_pi, nd));
    CK(down.copy(out->dyn_iskey, ctx->d_s_iskey, nd)); CK(down.copy(out->dyn_rep_read, ctx->d_s_rep_read, nd));
    CK(down.copy(out->dyn_rep_qpos, ctx->d_s_rep_qpos, nd)); CK(down.copy(out->dyn_len, ctx->d_s_len, nd));
    std::vector<unsigned long long> keys((size_t)nd);
    std::vector<uint32_t> first(nl + 1);
    CK(down.copy(keys.data(), ctx->d_s_key, nd)); CK(down.copy(first.data(), ctx->d_dyn_first, nl + 1));
    CK(cudaEventRecord(ctx->ev[EV_COPY_END], ctx->st));
    CK(cudaStreamSynchronize(ctx->st));
    for (int64_t j = 0; j < nd; ++j) {
        unsigned long long k = keys[(size_t)j];
        if (out->dyn_locus) out->dyn_locus[j] = (int32_t)(k >> DYN_LOCUS_SHIFT);
        if (out->dyn_kind) out->dyn_kind[j] = (uint8_t)((k >> 40) & 3u);
        if (out->dyn_site) out->dyn_site[j] = (uint8_t)((k >> 36) & 15u);
    }
    if (out->dyn_first) for (size_t i = 0; i <= nl; ++i) out->dyn_first[i] = first[i];
    cudaEventElapsedTime(&ctx->tm.ms_d2h, ctx->ev[EV_COPY_BEGIN], ctx->ev[EV_COPY_END]);
    ctx->tm.bytes_d2h = down.bytes;
    return SMC_OK;
}

// SMC_TIMELINE=1: one stderr line per smc_call_batch with the host enter / exit times and the device times of the stage
// events, all in ms since the first call of the process (how the calls of several contexts interleave on one GPU).
static std::mutex g_tl_mu;
static cudaEvent_t g_tl_base = nullptr;
static std::chrono::steady_clock::time_point g_tl_t0;
static double tl_host_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - g_tl_t0).count(); }

extern "C" int smc_call_batch(smc_ctx* ctx, const smc_reads_soa* reads, const smc_loci* loci, const smc_umi_keep* keep, smc_out* out) {
    static const bool timeline = [] { const char* ev = getenv("SMC_TIMELINE"); return ev && atoi(ev) != 0; }();
    double tl_enter = 0;
    if (timeline && ctx) {
        std::lock_guard<std::mutex> lk(g_tl_mu);
        if (!g_tl_base) {
            cudaSetDevice(ctx->device);
            cudaEventCreate(&g_tl_base); cudaEventRecord(g_tl_base, ctx->st); cudaEventSynchronize(g_tl_base);
            g_tl_t0 = std::chrono::steady_clock::now();
        }
        tl_enter = tl_host_ms();
    }
    struct TlExit {
        smc_ctx* c; bool on; double enter; float dev[8];
        ~TlExit() { if (on) fprintf(stderr, "[smc timeline] ctx %p host %.2f .. %.2f | dev: scalars %.2f chunks_done %.2f run %.2f prep_done %.2f sort_done %.2f pileup_done %.2f "
                                            "stats_done %.2f\n", (void*)c, enter, tl_host_ms(), dev[0], dev[1], dev[2], dev[3], dev[4], dev[5], dev[6]); }
    } tl{ctx, false, tl_enter, {}};
    // Bases and qualities (3/4 of the bytes) are uploaded in chunks on a second stream while the kernels that only need the
    // per-read scalars already run; the pileup kernels are launched per chunk as the data arrives (upload_impl,
    // smc_run_resident).  Whatever happens, no copy may still read the caller's buffers when this returns.
    int rc = upload_impl(ctx, reads, loci, keep, true);
    if (rc == SMC_OK) rc = smc_run_resident(ctx);
    if (ctx) {
        cudaError_t e1 = cudaStreamSynchronize(ctx->st_copy), e2 = cudaStreamSynchronize(ctx->st);
        if (rc == SMC_OK && (e1 != cudaSuccess || e2 != cudaSuccess)) {
            ctx->err = std::string("smc_call_batch: ") + cudaGetErrorString(e1 != cudaSuccess ? e1 : e2); rc = SMC_E_CUDA;
        }
        if (rc == SMC_OK && ctx->uploaded) cudaEventElapsedTime(&ctx->tm.ms_h2d, ctx->ev[EV_COPY_BEGIN], ctx->ev[EV_COPY_END]);
        if (timeline && rc == SMC_OK) {
            for (int i = EV_COPY_BEGIN; i <= EV_STATS_DONE; ++i) if (cudaEventElapsedTime(&tl.dev[i], g_tl_base, ctx->ev[i]) != cudaSuccess) { tl.dev[i] = -1.f; cudaGetLastError(); }
            tl.on = true;
        }
        ctx->pipe_n = 0;                                 // the batch is resident now: later smc_run_resident calls run it in one go
    }
    if (rc) return rc;
    return smc_download(ctx, out);
}

extern "C" int smc_host_alloc(int64_t bytes, void** out) {
    if (!out || bytes < 0) return SMC_E_ARG;
    *out = nullptr;
    cudaError_t e = cudaHostAlloc(out, (size_t)(bytes ? bytes : 1), cudaHostAllocPortable);
    if (e != cudaSuccess) { g_create_error = std::string("smc_host_alloc: ") + cudaGetErrorString(e); cudaGetLastError(); *out = nullptr; return SMC_E_CUDA; }
    return SMC_OK;
}

extern "C" void smc_host_free(void* p) { if (p) cudaFreeHost(p); }

extern "C" int smc_get_timings(smc_ctx* ctx, smc_timings* t) {
    if (!ctx || !t) return SMC_E_ARG;
    *t = ctx->tm;
    return SMC_OK;
}

extern "C" int smc_list_barcodes(smc_ctx* ctx, int64_t n, const int64_t* locus, int64_t* off_out, uint64_t* umi_out,
                                 uint32_t* first_read_out, int64_t umi_capacity) {
    if (!ctx) return SMC_E_ARG;
    if (!ctx->ran) { ctx->err = "smc_list_barcodes: run a batch first"; return SMC_E_STATE; }
    if (n < 0 || (n > 0 && (!locus || !off_out))) { ctx->err = "smc_list_barcodes: bad arguments"; return SMC_E_ARG; }
    CK(cudaSetDevice(ctx->device));
    const int64_t nl = ctx->n_loci;
    std::vector<int32_t> nbc((size_t)(nl ? nl : 1));
    if (nl)
        if (const int rc = read_back(ctx, nbc.data(), ctx->d_loc.as<int32_t>() + (size_t)SMC_L_NBC * nl, (size_t)nl * 4)) return rc;
    std::vector<int32_t> idx((size_t)(nl ? nl : 1), -1);
    off_out[0] = 0;
    for (int64_t k = 0; k < n; ++k) {
        if (locus[k] < 0 || locus[k] >= nl || (k > 0 && locus[k] <= locus[k - 1])) {
            ctx->err = "smc_list_barcodes: locus indices must be ascending and inside the batch"; return SMC_E_ARG;
        }
        idx[(size_t)locus[k]] = (int32_t)k;
        off_out[k + 1] = off_out[k] + nbc[(size_t)locus[k]];
    }
    const int64_t total = n ? off_out[n] : 0;
    if (total > umi_capacity || (total > 0 && (!umi_out || !first_read_out))) {
        ctx->err = "smc_list_barcodes: umi_capacity too small (needed count is off_out[n])"; return SMC_E_LIMIT;
    }
    if (total == 0 || ctx->n_tile_events == 0) return SMC_OK;
    CK(ctx->d_list_idx.ensure((size_t)nl * 4)); CK(ctx->d_list_count.ensure((size_t)n * 4)); CK(ctx->d_list_off.ensure((size_t)(n + 1) * 8));
    CK(ctx->d_list_umi.ensure((size_t)total * 8)); CK(ctx->d_list_first.ensure((size_t)total * 4));
    CK(cudaMemcpyAsync(ctx->d_list_idx.p, idx.data(), (size_t)nl * 4, cudaMemcpyHostToDevice, ctx->st));
    CK(cudaMemcpyAsync(ctx->d_list_off.p, off_out, (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, ctx->st));
    CK(cudaMemsetAsync(ctx->d_list_count.p, 0, (size_t)n * 4, ctx->st));
    // The listing pass re-runs the pileup kernel; it adds to the accumulators again, so the batch must be re-run
    // (with the mask) before the next download.
    ctx->ran = false;
    if (const int rc = ensure_code_storage(ctx, true, true)) return rc;
    KAArgs A; KBArgs B;
    fill_kargs(ctx, A, B, true, true);
    B.keep_idx = nullptr;
    B.list_idx = ctx->d_list_idx.as<int32_t>(); B.list_count = ctx->d_list_count.as<uint32_t>();
    B.list_off = ctx->d_list_off.as<int64_t>(); B.list_umi = ctx->d_list_umi.as<uint64_t>();
    B.list_first = ctx->d_list_first.as<uint32_t>(); B.list_cap = total;
    if (const int rc = launch_pileup<true>(ctx, A, B, false, false, nullptr)) return rc;
    CK(cudaMemcpyAsync(umi_out, ctx->d_list_umi.p, (size_t)total * 8, cudaMemcpyDeviceToHost, ctx->st));
    CK(cudaMemcpyAsync(first_read_out, ctx->d_list_first.p, (size_t)total * 4, cudaMemcpyDeviceToHost, ctx->st));
    CK(cudaStreamSynchronize(ctx->st));
    CK(cudaGetLastError());
    return SMC_OK;
}

extern "C" int smc_set_downsample(smc_ctx* ctx, int mode) {
    if (!ctx) return SMC_E_ARG;
    if (mode != SMC_DS_FLAG && mode != SMC_DS_DEVICE) { ctx->err = "smc_set_downsample: mode must be SMC_DS_FLAG or SMC_DS_DEVICE"; return SMC_E_ARG; }
    ctx->ds_mode = mode;
    return SMC_OK;
}

extern "C" int smc_set_barcode_hashes(smc_ctx* ctx, int64_t n, const uint64_t* code, const int64_t* py2_hash) {
    if (!ctx) return SMC_E_ARG;
    if (n < 0 || (n > 0 && (!code || !py2_hash))) { ctx->err = "smc_set_barcode_hashes: bad arguments"; return SMC_E_ARG; }
    for (int64_t i = 0; i < n; ++i)
        if (!(code[i] >> 63) || (i > 0 && code[i] <= code[i - 1])) {
            ctx->err = "smc_set_barcode_hashes: codes must be dictionary codes (top bit set), strictly ascending"; return SMC_E_ARG;
        }
    CK(cudaSetDevice(ctx->device));
    CK(ctx->d_bc_code.ensure((size_t)std::max<int64_t>(n, 1) * 8)); CK(ctx->d_bc_hash.ensure((size_t)std::max<int64_t>(n, 1) * 8));
    CK(cudaMemcpyAsync(ctx->d_bc_code.p, code, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->st));
    CK(cudaMemcpyAsync(ctx->d_bc_hash.p, py2_hash, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->st));
    CK(cudaStreamSynchronize(ctx->st));
    ctx->n_bc = n;
    return SMC_OK;
}

extern "C" int smc_draw_sample(smc_ctx* ctx, int64_t n_sets, const int64_t* off, const uint64_t* codes, const int64_t* seed_pos1,
                              const int64_t* k, int64_t* out) {
    if (!ctx) return SMC_E_ARG;
    if (n_sets < 0 || (n_sets > 0 && (!off || !seed_pos1 || !k || (off[n_sets] > 0 && (!codes || !out))))) {
        ctx->err = "smc_draw_sample: bad arguments"; return SMC_E_ARG;
    }
    if (n_sets == 0) return SMC_OK;
    for (int64_t i = 0; i < n_sets; ++i)
        if (off[0] != 0 || off[i + 1] < off[i] || k[i] < 0 || k[i] > off[i + 1] - off[i] || seed_pos1[i] < 0) {
            ctx->err = "smc_draw_sample: set " + std::to_string(i) + ": off must start at 0 and not decrease, 0 <= k <= set size, seed_pos1 >= 0";
            return SMC_E_ARG;
        }
    const int64_t T = off[n_sets];
    if (T > 0xffffffffll) { ctx->err = "smc_draw_sample: more than 2^32 keys"; return SMC_E_LIMIT; }
    CK(cudaSetDevice(ctx->device));
    const size_t tz = (size_t)(T ? T : 1);
    CK(ctx->d_list_off.ensure((size_t)(n_sets + 1) * 8)); CK(ctx->d_ds_k0.ensure((size_t)n_sets * 8)); CK(ctx->d_ds_k1.ensure((size_t)n_sets * 8));
    CK(ctx->d_list_umi.ensure(tz * 8)); CK(ctx->d_ds_v0.ensure(tz * 4));
    CK(cudaMemcpyAsync(ctx->d_list_off.p, off, (size_t)(n_sets + 1) * 8, cudaMemcpyHostToDevice, ctx->st));
    CK(cudaMemcpyAsync(ctx->d_ds_k0.p, seed_pos1, (size_t)n_sets * 8, cudaMemcpyHostToDevice, ctx->st));
    CK(cudaMemcpyAsync(ctx->d_ds_k1.p, k, (size_t)n_sets * 8, cudaMemcpyHostToDevice, ctx->st));
    CK(cudaMemcpyAsync(ctx->d_list_umi.p, codes, (size_t)T * 8, cudaMemcpyHostToDevice, ctx->st));
    uint64_t code_or = 0;
    if (const int rc = hash_barcodes(ctx, nullptr, ctx->d_list_umi.as<uint64_t>(), T, &code_or)) return rc;
    if (const int rc = draw_sets(ctx, ctx->d_list_off.as<int64_t>(), off, n_sets, T, ctx->d_ds_k0.as<int64_t>(), nullptr,
                                 ctx->d_ds_k1.as<int64_t>(), 0, ctx->d_ds_hash.as<int64_t>(), ctx->d_ds_v0.as<uint32_t>())) return rc;
    std::vector<uint32_t> idx(tz);
    if (const int rc = read_back(ctx, idx.data(), ctx->d_ds_v0.p, (size_t)T * 4)) return rc;
    CK(cudaGetLastError());
    for (int64_t i = 0; i < n_sets; ++i)
        for (int64_t j = 0; j < k[i]; ++j) out[off[i] + j] = idx[(size_t)(off[i] + j)];
    return SMC_OK;
}

extern "C" int smc_fisher_exact(smc_ctx* ctx, int64_t n, const int32_t* tables, double* p_out, double* or_out) {
    if (!ctx) return SMC_E_ARG;
    if (n < 0 || (n > 0 && (!tables || !p_out || !or_out))) { ctx->err = "smc_fisher_exact: bad arguments"; return SMC_E_ARG; }
    if (n == 0) return SMC_OK;
    for (int64_t i = 0; i < 4 * n; ++i) if (tables[i] < 0) { ctx->err = "smc_fisher_exact: negative cell"; return SMC_E_ARG; }
    CK(cudaSetDevice(ctx->device));
    CK(ctx->d_hp_bases.ensure((size_t)n * 16)); CK(ctx->d_hp_meta.ensure((size_t)n * 16));      // the candidate buffers double as scratch
    CK(cudaMemcpyAsync(ctx->d_hp_bases.p, tables, (size_t)n * 16, cudaMemcpyHostToDevice, ctx->st));
    double* dp = ctx->d_hp_meta.as<double>();
    k_fisher_tables<<<nblk(n * 32, 128), 128, 0, ctx->st>>>(ctx->d_hp_bases.as<int32_t>(), n, (int)ctx->prm.fisherLegacy, dp, dp + n);
    CK(cudaMemcpyAsync(p_out, dp, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->st));
    CK(cudaMemcpyAsync(or_out, dp + n, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->st));
    CK(cudaStreamSynchronize(ctx->st));
    CK(cudaGetLastError());
    return SMC_OK;
}

extern "C" int smc_hp_lowcomp(smc_ctx* ctx, const smc_hp_batch* Bt, uint8_t* flags_out) {
    if (!ctx) return SMC_E_ARG;
    if (!Bt || Bt->n < 0 || Bt->hpLen < 0 || (Bt->n > 0 && (!flags_out || !Bt->bases || !Bt->win_off || !Bt->win_len || !Bt->win_pos ||
                                                             !Bt->ref_off || !Bt->ref_len || !Bt->alt_off || !Bt->alt_len))) {
        ctx->err = "smc_hp_lowcomp: bad arguments"; return SMC_E_ARG;
    }
    const int64_t n = Bt->n;
    if (n == 0) return SMC_OK;
    for (int64_t k = 0; k < n; ++k) {                          // the kernel trusts these
        const bool ok = Bt->win_len[k] >= 0 && Bt->win_pos[k] >= 0 && Bt->win_pos[k] <= Bt->win_len[k] && Bt->ref_len[k] >= 0 &&
                        Bt->alt_len[k] >= 0 && Bt->win_off[k] >= 0 && Bt->win_off[k] + Bt->win_len[k] <= Bt->n_bases &&
                        Bt->ref_off[k] >= 0 && Bt->ref_off[k] + Bt->ref_len[k] <= Bt->n_bases && Bt->alt_off[k] >= 0 &&
                        Bt->alt_off[k] + Bt->alt_len[k] <= Bt->n_bases;
        if (!ok) { ctx->err = "smc_hp_lowcomp: candidate " + std::to_string(k) + " points outside bases[]"; return SMC_E_ARG; }
    }
    CK(cudaSetDevice(ctx->device));
    // device layout of the per-candidate metadata: three int64 arrays, then four int32 arrays
    const size_t n8 = (size_t)n * 8, n4 = (size_t)n * 4;
    CK(ctx->d_hp_bases.ensure((size_t)Bt->n_bases + 16)); CK(ctx->d_hp_meta.ensure(3 * n8 + 4 * n4)); CK(ctx->d_hp_flags.ensure((size_t)n));
    uint8_t* m = ctx->d_hp_meta.as<uint8_t>();
    CK(cudaMemcpyAsync(ctx->d_hp_bases.p, Bt->bases, (size_t)Bt->n_bases, cudaMemcpyHostToDevice, ctx->st));
    CK(cudaMemcpyAsync(m, Bt->win_off, n8, cudaMemcpyHostToDevice, ctx->st));
    CK(cudaMemcpyAsync(m + n8, Bt->ref_off, n8, cudaMemcpyHostToDevice, ctx->st));
    CK(cudaMemcpyAsync(m + 2 * n8, Bt->alt_off, n8, cudaMemcpyHostToDevice, ctx->st));
    CK(cudaMemcpyAsync(m + 3 * n8, Bt->win_len, n4, cudaMemcpyHostToDevice, ctx->st));
    CK(cudaMemcpyAsync(m + 3 * n8 + n4, Bt->win_pos, n4, cudaMemcpyHostToDevice, ctx->st));
    CK(cudaMemcpyAsync(m + 3 * n8 + 2 * n4, Bt->ref_len, n4, cudaMemcpyHostToDevice, ctx->st));
    CK(cudaMemcpyAsync(m + 3 * n8 + 3 * n4, Bt->alt_len, n4, cudaMemcpyHostToDevice, ctx->st));
    k_hp_lowcomp<<<nblk(n * 32, 128), 128, 0, ctx->st>>>(n, Bt->hpLen, ctx->d_hp_bases.as<uint8_t>(), (const int64_t*)m,
        (const int32_t*)(m + 3 * n8), (const int32_t*)(m + 3 * n8 + n4), (const int64_t*)(m + n8), (const int32_t*)(m + 3 * n8 + 2 * n4),
        (const int64_t*)(m + 2 * n8), (const int32_t*)(m + 3 * n8 + 3 * n4), ctx->d_hp_flags.as<uint8_t>());
    CK(cudaMemcpyAsync(flags_out, ctx->d_hp_flags.p, (size_t)n, cudaMemcpyDeviceToHost, ctx->st));
    CK(cudaStreamSynchronize(ctx->st));
    CK(cudaGetLastError());
    return SMC_OK;
}

// ------------------------------------------------------------------------------------------------------------
// BAM decode on the device (include/smc_b200.h: smc_decode_bam)
// ------------------------------------------------------------------------------------------------------------
// Device bytes a decode may need: the compressed and inflated streams, the scratch of partly kept blocks, about 200 bytes of
// per-record tables (at most one record per 36 stream bytes) and the output, which is no larger than the stream plus 64 bytes
// per record
static int64_t bam_decode_bytes(int64_t comp, int64_t raw, int64_t scratch) {
    const int64_t nrec = raw / 36 + 1;
    return comp + 64 + 2 * raw + scratch + nrec * 264 + ((int64_t)1 << 24);
}

static int bam_rewalk(smc_ctx* ctx, const uint8_t* raw, int64_t size, int64_t first, const BgzfJob* jobs, int64_t nb, int32_t nref,
                      int64_t t, int64_t start, std::vector<int64_t>& wk) {
    int64_t* d = ctx->d_bz_walk.as<int64_t>();
    CK(cudaMemcpyAsync(d + t, &start, 8, cudaMemcpyHostToDevice, ctx->st));
    k_walk<<<1, 1, 0, ctx->st>>>(raw, size, first, jobs, nb, t, t + 1, nref, 0, d, nullptr, nullptr);
    ++g_launches;
    for (int k = 0; k < 4; ++k) CK(cudaMemcpyAsync(&wk[(size_t)k * nb + t], d + (size_t)k * nb + t, 8, cudaMemcpyDeviceToHost, ctx->st));
    CK(cudaStreamSynchronize(ctx->st));
    return SMC_OK;
}

extern "C" int smc_decode_bam(smc_ctx* ctx, const smc_bgzf_block* blocks, int64_t n_blocks, const uint8_t* comp, int64_t comp_bytes,
                              int64_t raw_bytes, int64_t first_record, int32_t n_ref, int64_t n_iv, const int32_t* iv_ref,
                              const int32_t* iv_start, const int32_t* iv_end, int32_t trim, smc_bam_reads* out) {
    if (!ctx) return SMC_E_ARG;
    if (!out || n_blocks < 0 || comp_bytes < 0 || raw_bytes < 0 || n_ref < 0 || first_record < 0 || (n_blocks > 0 && (!blocks || !comp)) ||
        (n_iv > 0 && (!iv_ref || !iv_start || !iv_end))) {
        ctx->err = "smc_decode_bam: bad argument"; return SMC_E_ARG;
    }
    NvtxRange nv("smc_decode_bam");
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->st;
    const bool timing = getenv("SMC_BAM_TIMING") != nullptr;
    constexpr int NEV = 10;
    cudaEvent_t ev[NEV];
    for (auto& e : ev) CK(cudaEventCreate(&e));
    struct EvFree { cudaEvent_t* e; ~EvFree() { for (int k = 0; k < NEV; ++k) cudaEventDestroy(e[k]); } } ev_free{ev};
    // the block table: validated against the streams, and the scratch offset of every block that is only partly kept
    std::vector<BgzfJob> jobs((size_t)n_blocks);
    int64_t scratch = 0, uoff = 0;
    for (int64_t i = 0; i < n_blocks; ++i) {
        const smc_bgzf_block& b = blocks[i];
        if (b.coff < 0 || b.clen < 0 || b.coff + b.clen > comp_bytes || b.lo > b.hi || b.hi > b.isize || b.uoff != uoff) {
            ctx->err = "smc_decode_bam: block " + std::to_string(i) + " does not fit the compressed or the inflated stream"; return SMC_E_ARG;
        }
        const bool whole = b.lo == 0 && b.hi == b.isize;
        jobs[(size_t)i] = BgzfJob{b.coff, b.clen, b.uoff, whole ? 0 : scratch, b.isize, b.lo, b.hi, whole ? 1u : 0u};
        if (!whole) scratch += b.isize;
        uoff += b.hi - b.lo;
    }
    if (uoff != raw_bytes || first_record > raw_bytes) { ctx->err = "smc_decode_bam: the blocks do not add up to raw_bytes"; return SMC_E_ARG; }
    {   // what the device can hold: streams of up to 4 GiB (32-bit scans) that fit the free memory
        size_t free_b = 0, total_b = 0;
        CK(cudaMemGetInfo(&free_b, &total_b));
        int64_t budget = (int64_t)free_b;
        if (const char* ev_b = getenv("SMC_BAM_DEVICE_BUDGET")) budget = std::min<int64_t>(budget, atoll(ev_b));
        const int64_t need = bam_decode_bytes(comp_bytes, raw_bytes, scratch);
        if (raw_bytes >= ((int64_t)1 << 32) || need > budget) {
            ctx->err = "smc_decode_bam: the inflated stream (" + std::to_string(raw_bytes) + " bytes, about " + std::to_string(need >> 20) +
                       " MiB of device memory) exceeds the device budget (" + std::to_string(budget >> 20) + " MiB, streams < 4 GiB)";
            return SMC_E_BUDGET;
        }
    }
    const int64_t nb = n_blocks;
    CK(ctx->d_bz_comp.ensure((size_t)comp_bytes + 64));
    CK(ctx->d_bz_jobs.ensure(sizeof(BgzfJob) * (size_t)(nb + 1)));
    CK(ctx->d_bz_raw.ensure((size_t)raw_bytes + 64));
    CK(ctx->d_bz_scratch.ensure((size_t)scratch + 64));
    CK(ctx->d_bz_status.ensure(4 * (size_t)(nb + 1)));
    CK(ctx->d_bz_walk.ensure(32 * (size_t)(nb + 1)));
    CK(ctx->d_bz_base.ensure(8 * (size_t)(nb + 1)));
    CK(ctx->d_bz_small.ensure(256));
    uint8_t* raw = ctx->d_bz_raw.as<uint8_t>();
    BgzfJob* d_jobs = ctx->d_bz_jobs.as<BgzfJob>();
    uint32_t* small = ctx->d_bz_small.as<uint32_t>();             // [0, 1] bad record (u64), 2 any_dict, 4.. scan totals
    CK(cudaEventRecord(ev[0], st));
    if (comp_bytes) CK(cudaMemcpyAsync(ctx->d_bz_comp.p, comp, (size_t)comp_bytes + 64, cudaMemcpyHostToDevice, st));
    if (nb) CK(cudaMemcpyAsync(d_jobs, jobs.data(), sizeof(BgzfJob) * (size_t)nb, cudaMemcpyHostToDevice, st));
    CK(cudaEventRecord(ev[1], st));
    // ---- inflate
    LAUNCH(k_inflate, nblk(nb, INFLATE_WARPS), INFLATE_WARPS * 32, 0, ctx->d_bz_comp.as<uint8_t>(), d_jobs, nb, raw,
           ctx->d_bz_scratch.as<uint8_t>(), ctx->d_bz_status.as<int32_t>(), 1);
    CK(cudaGetLastError());
    CK(cudaEventRecord(ev[2], st));
    // ---- record boundaries
    int64_t* d_wk = ctx->d_bz_walk.as<int64_t>();
    LAUNCH(k_walk, nblk(nb, 128), 128, 0, raw, raw_bytes, first_record, d_jobs, nb, (int64_t)0, nb, n_ref, 1, d_wk, (int64_t*)nullptr,
           (const int64_t*)nullptr);
    std::vector<int32_t> status((size_t)nb);
    std::vector<int64_t> wk(4 * (size_t)nb);
    if (nb) {
        CK(cudaMemcpyAsync(status.data(), ctx->d_bz_status.p, 4 * (size_t)nb, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(wk.data(), d_wk, 32 * (size_t)nb, cudaMemcpyDeviceToHost, st));
    }
    CK(cudaStreamSynchronize(st));
    for (int64_t i = 0; i < nb; ++i)
        if (status[(size_t)i] != 0) {
            ctx->err = "smc_decode_bam: the device inflater rejects BGZF block " + std::to_string(i) + " (compressed offset " +
                       std::to_string(blocks[i].coff) + ")";
            return SMC_E_INFLATE;
        }
    // every range must start where the previous one ended (the first at the first record): by induction the chain is then the
    // true one; a range that does not is walked again from there
    std::vector<int64_t> base((size_t)nb + 1, 0);
    {
        int64_t expect = first_record;
        for (int64_t t = 0; t < nb; ++t) {
            if (wk[(size_t)t] != expect) { const int rc = bam_rewalk(ctx, raw, raw_bytes, first_record, d_jobs, nb, n_ref, t, expect, wk); if (rc) return rc; }
            if (wk[(size_t)(3 * nb + t)] >= 0) { ctx->err = "truncated BAM record at offset " + std::to_string(wk[(size_t)(3 * nb + t)]); return SMC_E_ARG; }
            expect = wk[(size_t)(nb + t)];
            base[(size_t)t + 1] = base[(size_t)t] + wk[(size_t)(2 * nb + t)];
        }
    }
    const int64_t nrec = base[(size_t)nb];
    CK(ctx->d_bz_offs.ensure(8 * (size_t)(nrec + 1)));
    if (nb) CK(cudaMemcpyAsync(ctx->d_bz_base.p, base.data(), 8 * (size_t)nb, cudaMemcpyHostToDevice, st));
    LAUNCH(k_walk, nblk(nb, 128), 128, 0, raw, raw_bytes, first_record, d_jobs, nb, (int64_t)0, nb, n_ref, 0, d_wk, ctx->d_bz_offs.as<int64_t>(),
           ctx->d_bz_base.as<int64_t>());
    CK(cudaEventRecord(ev[3], st));
    // ---- fields
    const smc_rec::Targets tg((size_t)n_ref, n_iv, iv_ref, iv_start, iv_end);
    const size_t ntg = tg.st.size();
    std::vector<int64_t> tgv(tg.off.begin(), tg.off.end());
    tgv.insert(tgv.end(), tg.st.begin(), tg.st.end());
    tgv.insert(tgv.end(), tg.en.begin(), tg.en.end());
    CK(ctx->d_bz_tg.ensure(8 * tgv.size()));
    CK(cudaMemcpyAsync(ctx->d_bz_tg.p, tgv.data(), 8 * tgv.size(), cudaMemcpyHostToDevice, st));
    const int64_t* d_tg = ctx->d_bz_tg.as<int64_t>();
    CK(ctx->d_bz_info.ensure(sizeof(BamRec) * (size_t)(nrec + 1)));
    CK(ctx->d_bz_cnt.ensure(4 * 4 * (size_t)(nrec + 1)));
    CK(ctx->d_bz_k0.ensure(8 * (size_t)(nrec + 1))); CK(ctx->d_bz_k1.ensure(8 * (size_t)(nrec + 1)));
    CK(ctx->d_bz_v0.ensure(4 * (size_t)(nrec + 1))); CK(ctx->d_bz_v1.ensure(4 * (size_t)(nrec + 1)));
    CK(ctx->d_bz_first.ensure(4 * (size_t)(nrec + 1))); CK(ctx->d_bz_isfirst.ensure(4 * (size_t)(nrec + 1)));
    CK(ctx->d_bz_hist.ensure(4 * radix_hist_words(nrec)));
    CK(ctx->d_bz_scan.ensure(4 * (size_t)std::max<int64_t>(radix_scan_words(nrec), scan_scratch_words(4 * nrec))));
    const BamRec* info = ctx->d_bz_info.as<BamRec>();
    const int64_t* offs = ctx->d_bz_offs.as<int64_t>();
    uint32_t* cnt = ctx->d_bz_cnt.as<uint32_t>();
    CK(cudaMemsetAsync(small, 0xff, 8, st));
    CK(cudaMemsetAsync(small + 2, 0, 64, st));
    const int has_tg = n_iv > 0 ? 1 : 0, do_trim = trim && n_iv > 0 ? 1 : 0;
    LAUNCH(k_fields, nblk(nrec, 256), 256, 0, raw, raw_bytes, offs, nrec, n_ref, d_tg, d_tg + n_ref + 1, d_tg + n_ref + 1 + ntg, has_tg, do_trim,
           ctx->d_bz_info.as<BamRec>(), cnt, ctx->d_bz_k0.as<uint64_t>(), ctx->d_bz_v0.as<uint32_t>(), reinterpret_cast<unsigned long long*>(small),
           small + 2);
    CK(cudaGetLastError());
    CK(cudaEventRecord(ev[4], st));
    // ---- identities: records sorted stably by identity hash, the first of each identity verified on the name bytes, ids by a
    // scan over "is a first record" in record order; then the same for the barcodes that need the dictionary
    auto number = [&](uint32_t* first, uint32_t* isfirst, int bc_only, uint32_t* total) {
        const int r = radix_sort_bits<uint64_t>(ctx->d_bz_k0.as<uint64_t>(), ctx->d_bz_v0.as<uint32_t>(), ctx->d_bz_k1.as<uint64_t>(),
                                                ctx->d_bz_v1.as<uint32_t>(), nrec, 0, 64, ctx->d_bz_hist.as<uint32_t>(), ctx->d_bz_scan.as<uint32_t>(), st);
        cudaMemsetAsync(isfirst, 0, 4 * (size_t)(nrec + 1), st);
        LAUNCH(k_first, nblk(nrec, 256), 256, 0, r ? ctx->d_bz_k1.as<uint64_t>() : ctx->d_bz_k0.as<uint64_t>(),
               r ? ctx->d_bz_v1.as<uint32_t>() : ctx->d_bz_v0.as<uint32_t>(), nrec, raw, offs, info, bc_only, first, isfirst);
        exclusive_scan_u32(isfirst, first == ctx->d_bz_first.as<uint32_t>() ? ctx->d_bz_k1.as<uint32_t>() : ctx->d_bz_v1.as<uint32_t>(), nrec,
                           ctx->d_bz_scan.as<uint32_t>(), total, st);
    };
    // frag ids land in d_bz_k1 (viewed as u32) once the identity sort no longer needs it; dictionary ids in d_bz_v1
    number(ctx->d_bz_first.as<uint32_t>(), ctx->d_bz_isfirst.as<uint32_t>(), 0, small + 4);
    uint32_t any_dict = 0;
    CK(cudaMemcpyAsync(&any_dict, small + 2, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    uint32_t* fid = ctx->d_bz_k1.as<uint32_t>();
    uint32_t* dfirst = nullptr; uint32_t* did = nullptr; uint32_t* disfirst = nullptr;
    if (any_dict) {
        // the identity ids move out of d_bz_k1 before the dictionary sort reuses it
        CK(ctx->d_bz_disfirst.ensure(4 * (size_t)(nrec + 1)));
        CK(cudaMemcpyAsync(ctx->d_bz_isfirst.p, fid, 4 * (size_t)nrec, cudaMemcpyDeviceToDevice, st));
        fid = ctx->d_bz_isfirst.as<uint32_t>();
        CK(ctx->d_bz_dfirst.ensure(4 * (size_t)(nrec + 1)));
        LAUNCH(k_dict_keys, nblk(nrec, 256), 256, 0, raw, offs, nrec, info, ctx->d_bz_k0.as<uint64_t>(), ctx->d_bz_v0.as<uint32_t>());
        dfirst = ctx->d_bz_dfirst.as<uint32_t>(); disfirst = ctx->d_bz_disfirst.as<uint32_t>();
        number(dfirst, disfirst, 1, small + 5);
        did = ctx->d_bz_v1.as<uint32_t>();
    }
    CK(cudaGetLastError());
    CK(cudaEventRecord(ev[5], st));
    // ---- offsets: output slots and payload offsets (scans of the four counts), their totals, then the output arena
    for (int k = 0; k < 4; ++k) exclusive_scan_u32(cnt + (size_t)k * nrec, cnt + (size_t)k * nrec, nrec, ctx->d_bz_scan.as<uint32_t>(), small + 6 + k, st);
    CK(cudaEventRecord(ev[6], st));
    uint32_t tot[6] = {0, 0, 0, 0, 0, 0};                 // identities, dictionary barcodes, kept reads, seq bytes, quality bytes, CIGAR words
    unsigned long long bad = 0;
    CK(cudaMemcpyAsync(tot, small + 4, sizeof(tot), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&bad, small, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (bad != ~0ull) { ctx->err = "malformed BAM record (field lengths exceed block_size)"; return SMC_E_ARG; }
    const int64_t n = tot[2], ndict = any_dict ? tot[1] : 0;
    // the arena: every output array 256-byte aligned, in one device buffer and one pinned host buffer (one copy back)
    size_t at = 0;
    auto carve = [&](size_t bytes) { const size_t o = at; at += (bytes + 255) & ~(size_t)255; return o; };
    const size_t o_ref = carve(4 * n), o_pos = carve(4 * n), o_nm = carve(4 * n), o_lseq = carve(4 * n), o_slo = carve(do_trim ? 4 * n : 0),
                 o_slen = carve(do_trim ? 4 * n : 0), o_frag = carve(4 * n), o_flag = carve(2 * n), o_ncig = carve(2 * n), o_mapq = carve(n),
                 o_soff = carve(8 * n), o_qoff = carve(8 * n), o_coff = carve(8 * n), o_umi = carve(8 * n), o_cig = carve(4 * (size_t)tot[5]),
                 o_seq = carve(tot[3]), o_qual = carve(tot[4]), o_hist = carve(256 * 8);
    CK(ctx->d_bz_out.ensure(at));
    // Ordinary host memory: a decode is one copy back, and page-locking the arena cost 250-290 ms for a 100-interval panel on a
    // B200 host (profiles/bam_decode_gpu_b200.jsonl) against about 12 ms for the copy itself
    if (ctx->h_bz_cap < at) {
        free(ctx->h_bz_out);
        ctx->h_bz_out = malloc(at ? at : 1);
        if (!ctx->h_bz_out) { ctx->h_bz_cap = 0; ctx->err = "smc_decode_bam: out of host memory for the decoded arrays"; return SMC_E_CUDA; }
        ctx->h_bz_cap = at;
    }
    CK(cudaEventRecord(ev[7], st));           // ev[6] .. ev[7]: the totals' round trip and the output arena's allocation (host)
    uint8_t* D = ctx->d_bz_out.as<uint8_t>();
    uint8_t* H = static_cast<uint8_t*>(ctx->h_bz_out);
    BamOut o;
    o.ref_id = (int32_t*)(D + o_ref); o.pos = (int32_t*)(D + o_pos); o.nm = (int32_t*)(D + o_nm); o.l_seq = (int32_t*)(D + o_lseq);
    o.store_lo = (int32_t*)(D + o_slo); o.store_len = (int32_t*)(D + o_slen); o.frag_id = (uint32_t*)(D + o_frag);
    o.flag = (uint16_t*)(D + o_flag); o.n_cigar = (uint16_t*)(D + o_ncig); o.mapq = D + o_mapq; o.seq_off = (int64_t*)(D + o_soff);
    o.qual_off = (int64_t*)(D + o_qoff); o.cigar_off = (int64_t*)(D + o_coff); o.umi = (uint64_t*)(D + o_umi); o.cigar = D + o_cig;
    o.seq = D + o_seq; o.qual = D + o_qual; o.qual_hist = (unsigned long long*)(D + o_hist);
    o.n = n; o.seq_bytes = tot[3]; o.qual_bytes = tot[4]; o.cigar_words = tot[5];
    CK(cudaMemsetAsync(o.qual_hist, 0, 256 * 8, st));
    if (ndict) {
        CK(ctx->d_bz_dict.ensure((size_t)ndict * (BAM_DICT_STRIDE + 4)));
        LAUNCH(k_dict_strings, nblk(nrec, 256), 256, 0, raw, offs, nrec, info, disfirst, did, ctx->d_bz_dict.as<uint8_t>(),
               reinterpret_cast<uint32_t*>(ctx->d_bz_dict.as<uint8_t>() + (size_t)ndict * BAM_DICT_STRIDE));
    }
    LAUNCH(k_copy, (unsigned)std::min<int64_t>(nblk(nrec, COPY_WARPS), (int64_t)ctx->n_sm * 32), COPY_WARPS * 32, 0, raw, offs, nrec, info, cnt, ctx->d_bz_first.as<uint32_t>(), fid, dfirst, did, do_trim, o);
    CK(cudaGetLastError());
    CK(cudaEventRecord(ev[8], st));
    CK(cudaMemcpyAsync(H, D, at, cudaMemcpyDeviceToHost, st));
    std::vector<uint8_t> dict;
    if (ndict) {
        dict.resize((size_t)ndict * (BAM_DICT_STRIDE + 4));
        CK(cudaMemcpyAsync(dict.data(), ctx->d_bz_dict.p, dict.size(), cudaMemcpyDeviceToHost, st));
    }
    CK(cudaEventRecord(ev[9], st));
    CK(cudaStreamSynchronize(st));
    ctx->bz_dict.clear();
    for (int64_t k = 0; k < ndict; ++k) {
        uint32_t len;
        memcpy(&len, &dict[(size_t)ndict * BAM_DICT_STRIDE + 4 * (size_t)k], 4);
        ctx->bz_dict.emplace_back(reinterpret_cast<const char*>(&dict[(size_t)k * BAM_DICT_STRIDE]), len);
    }
    if (timing) {
        static const char* stage[NEV - 1] = {"H2D compressed", "inflate", "record boundaries", "fields + hash", "fragment identities",
                                             "offsets", "totals + output arena (host)", "copy", "D2H"};
        for (int k = 0; k < NEV - 1; ++k) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, ev[k], ev[k + 1]);
            fprintf(stderr, "[smc_b200] bam decode %s: %.3f ms\n", stage[k], ms);
        }
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ev[0], ev[NEV - 1]);
        fprintf(stderr, "[smc_b200] bam decode total: %.3f ms (%lld blocks, %lld compressed bytes, %lld inflated, %lld records, %lld kept)\n", ms,
                (long long)nb, (long long)comp_bytes, (long long)raw_bytes, (long long)nrec, (long long)n);
    }
    *out = smc_bam_reads{};
    out->n_reads = n;
    out->ref_id = (const int32_t*)(H + o_ref); out->pos = (const int32_t*)(H + o_pos); out->flag = (const uint16_t*)(H + o_flag);
    out->mapq = H + o_mapq; out->nm = (const int32_t*)(H + o_nm); out->l_seq = (const int32_t*)(H + o_lseq);
    out->seq_off = (const int64_t*)(H + o_soff); out->qual_off = (const int64_t*)(H + o_qoff); out->cigar_off = (const int64_t*)(H + o_coff);
    out->n_cigar = (const uint16_t*)(H + o_ncig); out->umi = (const uint64_t*)(H + o_umi); out->frag_id = (const uint32_t*)(H + o_frag);
    out->seq = H + o_seq; out->seq_bytes = tot[3]; out->qual = H + o_qual; out->qual_bytes = tot[4];
    out->cigar = (const uint32_t*)(H + o_cig); out->n_cigar_words = tot[5]; out->n_dict_umis = ndict;
    out->store_lo = do_trim ? (const int32_t*)(H + o_slo) : nullptr; out->store_len = do_trim ? (const int32_t*)(H + o_slen) : nullptr;
    out->qual_hist = (const uint64_t*)(H + o_hist);
    // the results are in the pinned arena: the device side of the decode goes back to the pool (a context that keeps the arrays
    // alive for the rest of a run holds no device memory for them)
    for (DevBuf* b : {&ctx->d_bz_comp, &ctx->d_bz_jobs, &ctx->d_bz_raw, &ctx->d_bz_scratch, &ctx->d_bz_status, &ctx->d_bz_walk, &ctx->d_bz_base,
                      &ctx->d_bz_offs, &ctx->d_bz_info, &ctx->d_bz_cnt, &ctx->d_bz_k0, &ctx->d_bz_k1, &ctx->d_bz_v0, &ctx->d_bz_v1, &ctx->d_bz_first,
                      &ctx->d_bz_isfirst, &ctx->d_bz_dfirst, &ctx->d_bz_disfirst, &ctx->d_bz_hist, &ctx->d_bz_scan, &ctx->d_bz_tg, &ctx->d_bz_out,
                      &ctx->d_bz_dict, &ctx->d_bz_small})
        b->release();
    return SMC_OK;
}

extern "C" const char* smc_decoded_dict_umi(smc_ctx* ctx, int64_t i) {
    return (ctx && i >= 0 && i < (int64_t)ctx->bz_dict.size()) ? ctx->bz_dict[(size_t)i].c_str() : "";
}

// caller-given raw DEFLATE streams through the device inflater (a validation entry point, like smc_fisher_exact)
extern "C" int smc_inflate_device(smc_ctx* ctx, int64_t n, const uint8_t* in, int64_t in_bytes, const int64_t* in_off, const int64_t* in_len,
                                  uint8_t* out, int64_t out_bytes, const int64_t* out_off, const int64_t* out_len, int32_t* status) {
    if (!ctx) return SMC_E_ARG;
    if (n < 0 || in_bytes < 0 || out_bytes < 0 || (n > 0 && (!in || !in_off || !in_len || !out || !out_off || !out_len || !status))) {
        ctx->err = "smc_inflate_device: bad argument"; return SMC_E_ARG;
    }
    std::vector<BgzfJob> jobs((size_t)n);
    for (int64_t i = 0; i < n; ++i) {
        if (in_off[i] < 0 || in_len[i] < 0 || in_off[i] + in_len[i] + 64 > in_bytes || out_off[i] < 0 || out_len[i] < 0 ||
            out_len[i] > 0xffffffffll || out_off[i] + out_len[i] > out_bytes) {
            ctx->err = "smc_inflate_device: stream " + std::to_string(i) + " does not fit its buffers"; return SMC_E_ARG;
        }
        jobs[(size_t)i] = BgzfJob{in_off[i], in_len[i], out_off[i], 0, (uint32_t)out_len[i], 0u, (uint32_t)out_len[i], 1u};
    }
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->st;
    CK(ctx->d_bz_comp.ensure((size_t)in_bytes + 1));
    CK(ctx->d_bz_raw.ensure((size_t)out_bytes + 1));
    CK(ctx->d_bz_jobs.ensure(sizeof(BgzfJob) * (size_t)(n + 1)));
    CK(ctx->d_bz_status.ensure(4 * (size_t)(n + 1)));
    if (n == 0) return SMC_OK;
    CK(cudaMemcpyAsync(ctx->d_bz_comp.p, in, (size_t)in_bytes, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(ctx->d_bz_raw.p, out, (size_t)out_bytes, cudaMemcpyHostToDevice, st));     // whatever lies between the outputs stays
    CK(cudaMemcpyAsync(ctx->d_bz_jobs.p, jobs.data(), sizeof(BgzfJob) * (size_t)n, cudaMemcpyHostToDevice, st));
    LAUNCH(k_inflate, nblk(n, INFLATE_WARPS), INFLATE_WARPS * 32, 0, ctx->d_bz_comp.as<uint8_t>(), ctx->d_bz_jobs.as<BgzfJob>(), n,
           ctx->d_bz_raw.as<uint8_t>(), (uint8_t*)nullptr, ctx->d_bz_status.as<int32_t>(), 0);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, ctx->d_bz_raw.p, (size_t)out_bytes, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(status, ctx->d_bz_status.p, 4 * (size_t)n, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return SMC_OK;
}
