"""smCounter command line and ``main(args)`` with the reference's contract (smCounter.py:616-640, 645-909), running the
per-locus calling hot path on B200 GPUs through libsmc_b200.so.

Same parameters (bamFile, bedTarget, refGenome, mtDepth, rpb, minBQ, minMQ, hpLen, mismatchThr, mtDrop, maxMT, primerDist,
threshold, bedTandemRepeats, bedRepeatMaskerSubset, runPath, logFile, paramFile, nCPU, bedtoolsPath), same three output
files with the same columns, same return value (the PI threshold).  What changes underneath:

  * the BAM is decoded once into flat SoA buffers (smcounter_b200.bam) instead of once per locus through pysam;
  * ``Pool(nCPU).apply_async(vc_wrapper, ...)`` per locus (smCounter.py:683-685) becomes one batched
    ``GpuCaller.call`` per GPU over depth-balanced BED-interval shards (``--gpus``; ``--nCPU`` is accepted and only
    bounds the host threads of the BAM decoder);
  * bedtools (smCounter.py:700-710) is replaced by in-process interval arithmetic (smcounter_b200.repeats);
    ``--bedtoolsPath`` is accepted and ignored.

There is no CPU implementation of the calling path in this package: without libsmc_b200.so or without a CUDA device
``main`` raises.
"""
from __future__ import annotations

import argparse
import datetime
import os
import queue
import threading
from concurrent.futures import ThreadPoolExecutor

import numpy as np

from . import repeats, writers
from .bam import read_bam
from ._bamio import pack_upload
from .caller import GpuCaller, PinnedArena, VcParams
from .downsample import py2_string_hash
from .fasta import FastaFile
from .rows import device_hp_flags, emit_rows, headerAll, headerVariants
from .shard import ReadLocator, plan_batches, plan_shards, split_long_intervals
from .soa import umi_string
from .targets import build_loci, intervals_from_bed_lines

parser = None


def argParseInit():
    """smCounter.py:617-640, plus --gpus (how many B200s to shard the target over)."""
    global parser
    parser = argparse.ArgumentParser(description='Variant calling using molecular barcodes', fromfile_prefix_chars='@')
    parser.add_argument('--outPrefix', default=None, required=True, help='prefix for output files')
    parser.add_argument('--bamFile', default=None, required=True, help='BAM file')
    parser.add_argument('--bedTarget', default=None, required=True, help='BED file for target region')
    parser.add_argument('--mtDepth', default=None, required=True, type=int, help='Mean MT depth')
    parser.add_argument('--rpb', default=None, required=True, type=float, help='Mean read pairs per MT')
    parser.add_argument('--nCPU', type=int, default=1, help='number of CPUs to use in parallel')
    parser.add_argument('--minBQ', type=int, default=20, help='minimum base quality allowed for analysis')
    parser.add_argument('--minMQ', type=int, default=30, help='minimum mapping quality allowed for analysis')
    parser.add_argument('--hpLen', type=int, default=10, help='Minimum length for homopolymers')
    parser.add_argument('--mismatchThr', type=float, default=6.0, help='average number of mismatches per 100 bases allowed')
    parser.add_argument('--mtDrop', type=int, default=0, help='Drop MTs with lower than or equal to X reads.')
    parser.add_argument('--maxMT', type=int, default=0, help='Randomly downsample to X MTs (max number of MTs at any position). If set to 0 (default), maxMT = 2.0 * mean MT depth')
    parser.add_argument('--primerDist', type=int, default=2, help='filter variants that are within X bases to primer')
    parser.add_argument('--threshold', type=int, default=0, help='Minimum prediction index for a variant to be called. Must be non-negative. Typically ranges from 10 to 60. If set to 0 (default), smCounter will choose the appropriate cutoff based on the mean MT depth.')
    parser.add_argument('--refGenome', default='/qgen/home/rvijaya/downloads/alt_hap_masked_ref/ucsc.hg19.fasta')
    parser.add_argument('--bedTandemRepeats', default='/qgen/home/xuc/UCSC/simpleRepeat.bed', help='bed for UCSC tandem repeats')
    parser.add_argument('--bedRepeatMaskerSubset', default='/qgen/home/xuc/UCSC/SR_LC_SL.nochr.bed', help='bed for RepeatMasker simple repeats, low complexity, microsatellite regions')
    parser.add_argument('--bedtoolsPath', default='/qgen/bin/bedtools-2.25.0/bin/', help='path to bedtools (accepted for compatibility; interval arithmetic is done in-process)')
    parser.add_argument('--runPath', default=None, help='path to working directory')
    parser.add_argument('--logFile', default=None, help='log file')
    parser.add_argument('--paramFile', default=None, help='optional parameter file that contains the above paramters. if specified, this must be the only parameter, except for --logFile.')
    parser.add_argument('--gpus', type=int, default=1, help='number of B200 GPUs to shard the target over (BED intervals, balanced by depth)')
    parser.add_argument('--bamDecoder', choices=('host', 'gpu'), default='host', help='where the BAM is inflated and decoded: host (default, threaded C++) or gpu (the first GPU of the run; the same reads)')
    parser.add_argument('--fisherLegacy', type=int, default=0, help='1: two-sided Fisher p-values as scipy <= 1.6 computed them (epsilon = 1 - 1e-4, the scipy of the 2017 reference run); 0 (default): scipy >= 1.7')


# Page-locked upload buffers are expensive to create (the driver pins every page): they are kept for the life of the process
# and handed from one call_loci() to the next.
_ARENAS: "queue.SimpleQueue[PinnedArena]" = queue.SimpleQueue()


def _take_arena() -> PinnedArena:
    try:
        return _ARENAS.get_nowait()
    except queue.Empty:
        return PinnedArena()


def release_host_buffers():
    """Frees the pinned upload buffers kept between calls."""
    while True:
        try:
            _ARENAS.get_nowait().close()
        except queue.Empty:
            return


def _run_shards(reads, intervals, refs, prm: VcParams, gpus, devices, stage_times, batch_limits, emit_kw):
    """Shards the BED intervals over the GPUs, streams every shard through its GPU in batches, and turns each batch's device
    results into text with the native output stage (rows.emit_rows).  Returns {interval index: (EmittedRows, first row, end row)}."""
    import time
    chroms = reads.chroms
    devices = list(devices) if devices is not None else list(range(max(1, gpus)))
    t_plan = time.perf_counter()
    locator = ReadLocator(reads, chroms)
    # an interval above the library's per-batch limits (a whole-chromosome BED line, a very deep amplicon) is processed as
    # consecutive sub-intervals; the callers below see one entry per ORIGINAL interval again
    lim = dict(batch_limits or {})
    pieces = split_long_intervals(intervals, locator, max_loci=lim.get("max_loci", 1 << 20), max_payload_bytes=lim.get("max_payload_bytes", 1 << 30),
                                  max_reads=lim.get("max_reads", 1 << 27))
    if len(pieces) != len(intervals):
        sub = _run_shards(reads, pieces, refs, prm, gpus, devices, stage_times, batch_limits, emit_kw)
        return _regroup_pieces(intervals, pieces, sub)
    plan = plan_shards(reads, intervals, chroms, len(devices), locator)
    pack_threads = max(2, (os.cpu_count() or 2) // max(1, len(devices)))       # the shards of all GPUs pack side by side
    compactable = reads.qual_bits == 8 and reads.scalar_bits == 32 and reads.seq_bits == 4 and os.environ.get("SMC_NATIVE_PACK", "1") != "0"
    per_interval = {}
    errors = [None] * len(plan)
    lock = threading.Lock()
    if stage_times is not None:
        stage_times["ms_plan"] = stage_times.get("ms_plan", 0.0) + 1e3 * (time.perf_counter() - t_plan)

    def work(g):
        try:
            idxs = plan[g][0]
            if not idxs:
                return
            # a shard goes through its GPU as a stream of batches under the library's per-batch limits
            batches = plan_batches(locator, intervals, idxs, **(batch_limits or {}))
            # Up to three contexts and host threads per GPU: while one batch computes and another downloads, the next one is already uploading
            # (ctypes drops the GIL inside the library), so the PCIe link and the SMs are both kept busy across batches.
            n_ctx = max(1, min(int(os.environ.get("SMC_CTX_PER_GPU", "3")), len(batches)))
            t_create = time.perf_counter()
            callers = [GpuCaller(prm, devices[g], device_downsample=True) for _ in range(n_ctx)]      # smCounter.py:486-500 on the device
            arenas = [_take_arena() for _ in range(n_ctx)]      # the upload buffers of each context, recycled batch after batch
            free = queue.SimpleQueue()
            for i in range(n_ctx):
                free.put(i)
            if stage_times is not None:
                with lock:
                    stage_times["ms_ctx_create"] = stage_times.get("ms_ctx_create", 0.0) + 1e3 * (time.perf_counter() - t_create)

            def do_batch(b):
                i = free.get()
                try:
                    caller = callers[i]
                    ivs = [intervals[k] for k in b]
                    whole = len(plan) == 1 and len(batches) == 1
                    # the batch's reads, gathered and written in the compact wire encodings by one native pass (include/smc_soa.h)
                    arenas[i].reset()
                    t_pack = time.perf_counter()
                    if compactable:
                        sub = pack_upload(reads, None if whole else locator.select(ivs), alloc=arenas[i].take, threads=pack_threads)
                    else:
                        sub = reads if whole else reads.select(locator.select(ivs))
                    loci, bed_order = build_loci(ivs, chroms, refs)
                    t0 = time.perf_counter()
                    if stage_times is not None:
                        with lock:
                            stage_times["ms_select_pack"] = stage_times.get("ms_select_pack", 0.0) + 1e3 * (t0 - t_pack)
                    caller.set_barcode_hashes(*_dictionary_hashes(sub.umi, reads.umi_names))
                    res = caller.call(sub, loci)
                    tm = caller.timings()
                    hp = device_hp_flags(caller, res, sub, loci, chroms, refs, prm.hpLen)   # isHPorLowComp, smCounter.py:122-177
                    t1 = time.perf_counter()
                    em = emit_rows(res, sub, loci, chroms, refs, prm.hpLen, bed_order, hp_flags=hp, **emit_kw)
                    o = 0
                    with lock:
                        for k in b:
                            nrow = max(0, intervals[k][2] - intervals[k][1])
                            per_interval[k] = (em, o, o + nrow)
                            o += nrow
                        if stage_times is not None:
                            for key in ("ms_h2d", "ms_total_device", "ms_d2h"):
                                stage_times[key] = stage_times.get(key, 0.0) + float(tm[key])
                            stage_times["ms_gpu_call"] = stage_times.get("ms_gpu_call", 0.0) + 1e3 * (t1 - t0)
                            stage_times["ms_format_rows"] = stage_times.get("ms_format_rows", 0.0) + 1e3 * (time.perf_counter() - t1)
                            stage_times["batches"] = stage_times.get("batches", 0) + 1
                finally:
                    free.put(i)
            try:
                if n_ctx == 1:
                    for b in batches:
                        do_batch(b)
                else:
                    with ThreadPoolExecutor(max_workers=n_ctx) as ex:
                        for f in [ex.submit(do_batch, b) for b in batches]:
                            f.result()
            finally:
                for c in callers:
                    c.close()
                for a in arenas:
                    _ARENAS.put(a)
        except BaseException as e:          # noqa: BLE001 -- re-raised on the main thread
            errors[g] = e

    if len(plan) == 1:
        work(0)
    else:
        ts = [threading.Thread(target=work, args=(g,)) for g in range(len(plan))]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
    for e in errors:
        if e is not None:
            raise e
    return per_interval


def _dictionary_hashes(umi, names):
    """The batch's dictionary-coded barcodes (top bit set: not spelt by their code) and their Py2 string hashes, for the device
    draw of the down-sampling sample."""
    if umi.dtype != np.uint64:
        return np.zeros(0, np.uint64), np.zeros(0, np.int64)
    codes = np.unique(umi[umi >= np.uint64(1 << 63)])
    return codes, np.asarray([py2_string_hash(umi_string(int(c), names)) for c in codes], dtype=np.int64)


class _Joined:
    """Rows of several consecutive pieces of one BED interval, presented like one EmittedRows."""

    def __init__(self, parts):
        self.parts = parts                                   # [(EmittedRows, r0, r1)]

    def rows(self):
        out = []
        for em, r0, r1 in self.parts:
            out.extend(em.rows()[r0:r1])
        return out

    def slices(self, r0, r1):
        assert r0 == 0
        cols = ([], [], [])
        for em, a, b in self.parts:
            for dst, piece in zip(cols, em.slices(a, b)):
                dst.append(piece)
        return tuple(b"".join(c) for c in cols)


def _regroup_pieces(intervals, pieces, sub):
    """{piece index: rows} -> {original interval index: rows}: the pieces of an interval are consecutive and tile it."""
    out, j = {}, 0
    for k, (c, s, e) in enumerate(intervals):
        parts, pos = [], s
        while j < len(pieces) and pieces[j][0] == c and pieces[j][1] == pos and pieces[j][2] <= e and pos < e:
            if j in sub:
                parts.append(sub[j])
            pos = pieces[j][2]
            j += 1
        if e <= s and j < len(pieces) and pieces[j] == (c, s, e):
            j += 1
        if len(parts) == 1:
            out[k] = parts[0]
        elif parts:
            n = sum(r1 - r0 for (_, r0, r1) in parts)
            out[k] = (_Joined(parts), 0, n)
    return out


def call_loci(reads, intervals, refs, prm: VcParams, gpus: int = 1, devices=None, stage_times: dict | None = None,
              batch_limits: dict | None = None):
    """The drop-in for the reference's per-locus fan-out: rows of vc() (45 tab-joined fields each, FILTER still in
    accumulator form) for every position of ``intervals`` in BED order.

    ``reads``: ReadsSoA of the BAM; ``refs``: object with fetch()/get_reference_length().  One host thread per GPU
    (ctypes drops the GIL); a failing shard fails the run like smCounter.py:690-694.  ``stage_times`` (optional dict)
    receives the wall-clock ms of the device calls and of the row formatting, summed over shards.  A shard larger than
    the library's per-batch limits is streamed through its GPU in consecutive batches (``batch_limits``: keyword overrides
    of shard.plan_batches, for tests)."""
    per_interval = _run_shards(reads, intervals, refs, prm, gpus, devices, stage_times, batch_limits, {})
    cache, out = {}, []
    for k in range(len(intervals)):                    # BED order, like the reference's in-order p.get() (smCounter.py:685)
        if k in per_interval:
            em, r0, r1 = per_interval[k]
            rows = cache.get(id(em))
            if rows is None:
                rows = cache[id(em)] = em.rows()
            out.extend(rows[r0:r1])
    return out


def call_loci_text(reads, intervals, refs, prm: VcParams, threshold: int, trf=None, rm=None, gpus: int = 1, devices=None,
                   stage_times: dict | None = None, batch_limits: dict | None = None):
    """call_loci() + main()'s post-processing (repeat filters smCounter.py:751-785, PASS / strip, the called-variant rows of
    :832-891) in the native output stage: returns the bodies of the three output files (bytes, without their headers) in BED
    order: (all_txt, cut_txt, cut_vcf)."""
    per_interval = _run_shards(reads, intervals, refs, prm, gpus, devices, stage_times, batch_limits,
                               dict(finalize=True, threshold=threshold, trf=trf, rm=rm))
    parts = ([], [], [])
    for k in range(len(intervals)):
        if k in per_interval:
            em, r0, r1 = per_interval[k]
            for dst, piece in zip(parts, em.slices(r0, r1)):
                dst.append(piece)
    return tuple(b"".join(p) for p in parts)


def _read_track(path, flag, ncol):
    """A repeat track of main() (smCounter.py:699-710).  The reference hands the path to bedtools under check_call, so a
    missing file aborts the run; silently skipping it would report variants inside repeats as PASS.  Opting out is explicit:
    pass an empty string or 'none'."""
    if path is None or str(path).strip().lower() in ("", "none"):
        print("warning: %s disabled; its repeat filters (%s) are not applied" % (flag, "RepT" if ncol == 3 else "RepS/LowC/SL"))
        return []
    if not os.path.exists(path):
        raise IOError("%s: no such file: %r (the reference's bedtools call fails on a missing track; pass %s=none to run "
                      "without this filter)" % (flag, path, flag))
    return repeats.read_bed_rows(path, ncol) if ncol == 4 else repeats.read_bed_rows(path)


def main(args):
    timeStart = datetime.datetime.now()
    print("smCounter started at " + str(timeStart))
    if parser is None:
        argParseInit()
    if type(args) is not argparse.Namespace:                               # smCounter.py:656-660 (dict from a pipeline)
        argsList = []
        for argName, argVal in args.items():
            argsList.append("--{0}={1}".format(argName, argVal))
        args = parser.parse_args(argsList)
    elif args.paramFile is not None:                                       # :663-664
        args = parser.parse_args(("@" + args.paramFile,))
    for argName, argVal in vars(args).items():                             # :667-668
        print(argName, argVal)
    if args.runPath is not None:                                           # :671-672
        os.chdir(args.runPath)

    with open(args.bedTarget, 'r') as fh:                                  # :675-680
        bed_lines = fh.readlines()
    intervals = intervals_from_bed_lines(bed_lines)
    refs = FastaFile(args.refGenome)
    reads = read_bam(args.bamFile, intervals, threads=max(1, args.nCPU), trim=True,      # only the target windows cross PCIe
                     device=0 if getattr(args, 'bamDecoder', 'host') == 'gpu' else None)
    prm = VcParams(mtDepth=args.mtDepth, rpb=args.rpb, minBQ=args.minBQ, minMQ=args.minMQ, hpLen=args.hpLen,
                   mismatchThr=args.mismatchThr, mtDrop=args.mtDrop, maxMT=args.maxMT, primerDist=args.primerDist,
                   fisherLegacy=args.fisherLegacy)
    target_rows = [tuple(l.strip().split('\t')[0:3]) for l in bed_lines if not l.startswith("track ") and l.strip()]
    trf_rows = _read_track(args.bedTandemRepeats, "--bedTandemRepeats", 3)
    rm_rows = _read_track(args.bedRepeatMaskerSubset, "--bedRepeatMaskerSubset", 4)
    trf, rm = repeats.build_repeat_regions(target_rows, trf_rows, rm_rows)                # smCounter.py:699-734
    threshold = writers.pi_threshold(args.mtDepth, args.threshold)                         # :820
    try:
        # per-locus calling on the GPUs, then -- per batch, in the native output stage -- the rows, the repeat filters
        # (:751-785) and the called-variant lines (:832-891)
        all_txt, cut_txt, cut_vcf = call_loci_text(reads, intervals, refs, prm, threshold, trf, rm, gpus=args.gpus)
    except Exception as e:
        print(str(e))
        raise
    print("begin variant filtering and output")                           # :697
    with open(args.outPrefix + '.smCounter.all.txt', 'wb') as fh:          # :823-901
        fh.write(('\t'.join(headerAll) + '\n').encode()); fh.write(all_txt)
    with open(args.outPrefix + '.smCounter.cut.txt', 'wb') as fh:
        fh.write(('\t'.join(headerVariants) + '\n').encode()); fh.write(cut_txt)
    with open(args.outPrefix + '.smCounter.cut.vcf', 'wb') as fh:
        fh.write(writers.vcf_header(args.outPrefix).encode()); fh.write(cut_vcf)

    timeEnd = datetime.datetime.now()
    print("smCounter completed running at " + str(timeEnd))
    print("smCounter total time: " + str(timeEnd - timeStart))
    return threshold                                                       # :909


if __name__ == "__main__":
    argParseInit()
    _args = parser.parse_args()
    if _args.logFile:
        from . import run_log
        run_log.init(_args.logFile)
    main(_args)
