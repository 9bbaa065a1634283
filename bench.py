#!/usr/bin/env python
"""bench.py -- target loci called / s (BASELINE.json metric) on synthetic UMI-tagged panel reads, one process per GPU.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # the reference's own vc() on the host CPU (oracle/_ref)

Workload (``--workload``, default cfg2 = BASELINE.json configs[1]): seeded intervals of the N0030 panel BED, ~3 000 barcodes
per locus, ~4 read pairs per barcode, 2 x 150 bp.  A "step" is one pass of the hot path over one slice of the panel per GPU:
``--batches`` DISTINCT library batches of ``--intervals`` panel intervals each (every batch has its own reads and its own
pinned host buffers), streamed through the GPU one after the other -- so a timed region of K steps runs K x batches different
device calls, not the same batch K times.  ``value`` is measured with the batches resident in HBM (one context per batch),
``e2e`` through ``GpuCaller.call()`` + the device HP / LowC pass from pinned host buffers (H2D + kernels + D2H inside the timed
region, every step).  The panel is sharded across GPUs by BED interval (weak scaling: every rank gets its own slice); loci are
independent, so there is no data-path collective -- torch.distributed is used for the barrier and the max-over-ranks only.

The reads are a function of the arguments alone (not of the host's core count), so ``--dump-outputs DIR`` lets two builds be
compared output for output: after the timed steps it writes what the resident runs of the last step returned (see
``dump_outputs``) as float64 ``DIR/<name>.npy`` files.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PANEL_BED = os.path.join(ROOT, "tests", "golden", "n0030_panel.bed")
METRIC = "target_loci_called_per_sec"
UNIT = "loci/s"
ALGO_BYTES_PER_EVENT = 35.0     # SURVEY.md 8(d): reads in once (2.7 B/event) + every 16-byte event written once and read once
UMIS_PER_LOCUS, RPB = 3000, 4.0
SYNTH_GROUPS = 16               # make_panel_mp groups per batch: fixed, so that the reads do not depend on the host's core count
# --dump-outputs: a seeded sample of at most DUMP_LOCI loci (130 values each with the index and the non-finite codes) and DUMP_DYN
# of their dynamic-allele rows (20 values each), all float64: at most ~58 MB in all, under the DUMP_BYTES cap
DUMP_LOCI, DUMP_DYN, DUMP_BYTES = 40000, 100000, 64 * 10**6

# BASELINE.json configs as bench workloads: (description, SynthSpec keywords, VcParams keywords, default intervals per batch)
WORKLOADS = {
    "cfg2": ("cfg2 synthetic N0030 194-gene panel (primers...coding.bed geometry), 3000 UMIs/locus, rpb 4, 2x150bp",
             dict(umis_per_locus=3000, rpb=4.0, snv_every=1000, snv_vaf=0.01, indel_every=12000, indel_vaf=0.01),
             dict(mtDepth=3000, rpb=4.0, minBQ=20, minMQ=30, hpLen=10, mismatchThr=6.0, mtDrop=0, maxMT=0, primerDist=2), 96),
    "cfg1": ("cfg1 example-shaped (run.example.sh parameters): BRCA1 amplicon chr17:41243700-41245700 in 100-locus intervals, ~4100 UMIs/locus, 9.8 fragments/UMI",
             dict(umis_per_locus=5500, rpb=9.8, snv_every=250, snv_vaf=0.01, indel_every=600, indel_vaf=0.02),
             dict(mtDepth=3612, rpb=8.6, minBQ=20, minMQ=30, hpLen=8, mismatchThr=6.0, mtDrop=1, maxMT=0, primerDist=2), 5),
    "cfg3": ("cfg3 synthetic deep low-VAF panel: 150-bp amplicons, 20000 UMIs/locus, rpb 4, 0.5% VAF spike-ins every 50 bp",
             dict(umis_per_locus=20000, rpb=4.0, snv_every=50, snv_vaf=0.005),
             dict(mtDepth=20000, rpb=4.0, minBQ=20, minMQ=30, hpLen=10, mismatchThr=6.0, mtDrop=0, maxMT=0, primerDist=2), 8),
    "cfg5": ("cfg5 exome-scale shape: 200-bp intervals over 24 contigs, 1000 UMIs/locus, rpb 4, log-normal depth per interval (sigma 0.5)",
             dict(umis_per_locus=1000, rpb=4.0, snv_every=1000, snv_vaf=0.05, depth_sigma=0.5),
             dict(mtDepth=1000, rpb=4.0, minBQ=20, minMQ=30, hpLen=10, mismatchThr=6.0, mtDrop=0, maxMT=4000, primerDist=2), 320),
}


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=("b200", "reference"))
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--intervals", type=int, default=0, help="target intervals per library batch (0 = the workload's default; cfg2: 96)")
    ap.add_argument("--batches", type=int, default=8, help="distinct batches streamed per step and GPU")
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--cpu-loci", type=int, default=0, help="loci in the CPU-baseline sample (0 = 24 per core)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling leg (call_loci(gpus=N) on one fixed panel)")
    ap.add_argument("--whole-reads", action="store_true", help="upload whole reads instead of the target windows (store_lo/store_len)")
    ap.add_argument("--no-compact", action="store_true", help="upload one byte per quality and 32-bit scalars instead of the compact ABI v3 encodings")
    ap.add_argument("--pipeline-intervals", type=int, default=96,
                    help="intervals of the rank-0 batch run through the whole CLI path (BAM decode -> files); 0 = skip")
    ap.add_argument("--pipeline-repeats", type=int, default=5)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed resident runs of the last step returned to DIR/<name>.npy (float64)")
    a = ap.parse_args(argv)
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs needs --impl b200 (the reference arm returns text rows)")
    if a.intervals <= 0:
        a.intervals = WORKLOADS[a.workload][3]
    return a


def workload_intervals(args, world):
    """The intervals of the whole job: ``world * batches * intervals`` of them, in BED order."""
    from smcounter_b200.synth import panel_intervals_from_bed
    need = args.intervals * args.batches * world
    if args.workload == "cfg2":
        return panel_intervals_from_bed(PANEL_BED, limit=need, seed=args.seed)
    if args.workload == "cfg1":
        return [("chr17", 41243700 + 100 * k, 41243700 + 100 * (k + 1)) for k in range(need)]
    if args.workload == "cfg3":
        return [("chr%d" % (1 + k % 22), 100000 + 1000 * (k // 22), 100000 + 1000 * (k // 22) + 150) for k in range(need)]
    return [("chr%d" % (1 + k % 24), 100000 + 700 * (k // 24), 100000 + 700 * (k // 24) + 200) for k in range(need)]


def rank_batches(args, rank, world):
    """[intervals of batch 0, batch 1, ...] of this rank: the job's intervals go to ranks by the product's own multi-GPU plan
    (shard.assign_intervals: balanced by estimated work = interval length + a margin for the reads hanging over both ends; margin
    measured at N=4 on B200: 150 -> 5.14 ms max step, 300 -> 4.88, 600 -> 4.84), then to the rank's batches in BED order."""
    ivs = workload_intervals(args, world)
    if world > 1:
        from smcounter_b200.shard import assign_intervals
        margin = float(os.environ.get("SMC_BENCH_MARGIN", "500"))
        shard, _ = assign_intervals([float(e - s) + margin for (_, s, e) in ivs], world)
        ivs = [iv for iv, g in zip(ivs, shard) if g == rank]
    nb = args.batches
    cuts = [(len(ivs) * k) // nb for k in range(nb + 1)]
    return [ivs[cuts[k]:cuts[k + 1]] for k in range(nb)]


def _gen_batch(job):
    """One batch in a worker process: synthetic reads, trimmed to the targets and compacted (what the BAM decoder delivers)."""
    (ivs, spec_kw, seed, whole, no_compact, workers, keep_full) = job
    from smcounter_b200.synth import SynthSpec, make_panel_mp
    from smcounter_b200.targets import build_loci
    soa, refs, truth = make_panel_mp(ivs, SynthSpec(**spec_kw), seed=seed, workers=workers, n_groups=SYNTH_GROUPS)
    full = soa
    if not whole:
        soa = soa.trim_to_targets(ivs)
        if not no_compact:
            # 16-bit scalars, 2- / 4-bit quality codes + codebook, 2-bit bases + exception list (expanded on the device)
            soa = soa.compact(seq_bits_wanted=int(os.environ.get("SMC_BENCH_SEQ_BITS", "2")))
    loci, bed_order = build_loci(ivs, soa.chroms, refs)
    return ivs, soa, refs, loci, bed_order, (full if keep_full else None)


def make_batches(args, rank, world, only_first=False):
    """[(intervals, upload SoA, refs, loci, bed_order, whole-read SoA or None)] of this rank; generated by one worker process per
    batch (each with its share of the host cores)."""
    import pickle
    from concurrent.futures import ProcessPoolExecutor
    cache = os.environ.get("SMC_BENCH_CACHE")           # tuning sessions: reuse the generated batches between runs
    if cache:
        cache = "%s.%s_%d_%d_%d_%d_%d_%d%d%d" % (cache, args.workload, args.intervals, args.batches, args.seed, rank, world, int(args.whole_reads),
                                              int(args.no_compact), int(only_first))
        if os.path.exists(cache):
            with open(cache, "rb") as fh:
                return pickle.load(fh)
    groups = rank_batches(args, rank, world)
    if only_first:
        groups = groups[:1]
    spec_kw = WORKLOADS[args.workload][1]
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    per = max(1, min(16, cores // max(1, len(groups))))
    jobs = [(g, spec_kw, args.seed + 17 * rank + 1009 * k, args.whole_reads, args.no_compact, per, k == 0 and rank == 0) for k, g in enumerate(groups)]
    if len(jobs) == 1:
        out = [_gen_batch(jobs[0])]
    else:
        with ProcessPoolExecutor(max_workers=len(jobs)) as ex:
            out = list(ex.map(_gen_batch, jobs))
    if cache:
        with open(cache, "wb") as fh:
            pickle.dump(out, fh, protocol=4)
    return out


def vc_params(args=None):
    from smcounter_b200.caller import VcParams
    # cfg2 = SURVEY.md 8(d): --mtDepth 3000 --rpb 4.0 --mtDrop 0 --minBQ 20 --minMQ 30 --hpLen 10 (ds = 6000: no down-sampling)
    return VcParams(**WORKLOADS[args.workload if args is not None else "cfg2"][2])


def config_dict(args, world):
    """The ``config`` of the JSON line: identical for the CUDA arm and the reference arm (same workload, same loci)."""
    ivs = workload_intervals(args, world)
    p = WORKLOADS[args.workload][2]
    return {"workload": WORKLOADS[args.workload][0] + "; one step = %d distinct batches of %d intervals per GPU" % (args.batches, args.intervals),
            "intervals_per_batch": args.intervals, "batches_per_step": args.batches, "loci_per_step": int(sum(e - s for (_, s, e) in ivs)),
            "params": " ".join("%s %s" % kv for kv in p.items()), "seed": args.seed,
            "l2": "every step streams %d distinct batches (hundreds of MB each): inputs larger than L2, no flush needed" % args.batches,
            "parallelism": "panel sharded by BED interval (balanced by estimated events), no collective"}


def dump_outputs(path, outs, prefix="", share=1):
    """--dump-outputs: the LocusResults the resident runs of the last timed step downloaded, the rank's batches concatenated in
    batch order, as float64 ``path/<prefix><name>.npy``.  Per-locus arrays keep their layout (locus axis last) for a seeded sample
    of at most DUMP_LOCI / share loci, whose indices into the concatenation are ``locus``; the dynamic-allele rows of those loci
    (at most DUMP_DYN / share, a seeded sample beyond that) carry the same index in ``dyn_locus``.  Left out: dyn_rep_read /
    dyn_rep_qpos, which point at whichever read carrying the allele reached the device table first, so they vary from run to run.
    Every file holds finite numbers only: the floating-point results (PI, Fisher p and odds ratio; NaN where a test was not
    evaluated or an odds ratio is 0/0, +inf where it divides by zero) hold 0 in place of a non-finite value, and beside each
    ``<name>`` a ``<name>_nonfinite`` array of the same shape says which value it was: 0 finite, 1 +inf, -1 -inf, 2 NaN."""
    import numpy as np
    per_locus = ("loc", "cnt", "pi", "max_allele", "second_allele", "alt_allele", "alt_pi", "second_pi", "fl1", "fl2", "biallelic",
                 "fisher_p", "fisher_or")
    per_dyn = ("dyn_kind", "dyn_site", "dyn_len", "dyn_iskey", "dyn_cnt", "dyn_pi")
    base = np.cumsum([0] + [o.n_loci for o in outs])
    n, max_loci, max_dyn = int(base[-1]), DUMP_LOCI // share, DUMP_DYN // share
    rng = np.random.default_rng(0)
    locus = np.arange(n) if n <= max_loci else np.sort(rng.choice(n, size=max_loci, replace=False))
    arrays = {"locus": locus}
    for f in per_locus:
        arrays[f] = np.concatenate([getattr(o, f)[..., :o.n_loci] for o in outs], axis=-1)[..., locus]
    dyn_locus = np.concatenate([o.dyn_locus[:o.n_dyn].astype(np.int64) + b for o, b in zip(outs, base)])
    rows = np.flatnonzero(np.isin(dyn_locus, locus))
    if len(rows) > max_dyn:
        rows = np.sort(rng.choice(rows, size=max_dyn, replace=False))
    arrays["dyn_locus"] = dyn_locus[rows]
    for f in per_dyn:
        arrays[f] = np.concatenate([getattr(o, f)[:o.n_dyn] for o in outs])[rows]
    for k in [k for k, v in arrays.items() if v.dtype.kind == "f"]:
        v = arrays[k]
        code = np.where(np.isnan(v), 2.0, np.where(np.isinf(v), np.sign(v), 0.0))
        arrays[k], arrays[k + "_nonfinite"] = np.where(code == 0, v, 0.0), code
    arrays = {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in arrays.items()}
    assert all(np.isfinite(a).all() for a in arrays.values())
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_BYTES // share, total
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, prefix + k + ".npy"), a)
    return total


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md 'clocks' line): NVML every 5 ms when
    nvidia_ml_py is importable (the timed region is only a few hundred ms), else nvidia-smi every ~0.1 s."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        super().__init__(daemon=True)
        self.device = device
        self.sm, self.mx, self.reasons = [], [], set()
        self.stop_flag = False
        self.source = "nvidia-smi"

    def _run_nvml(self):
        import pynvml as nv
        nv.nvmlInit()
        # torch's device index follows CUDA_VISIBLE_DEVICES; NVML's does not
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = self.device
        if vis:
            try:
                idx = int(vis.split(",")[self.device])
            except Exception:
                pass
        h = nv.nvmlDeviceGetHandleByIndex(idx)
        self.mx.append(float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)))
        names = (("hw_slowdown", nv.nvmlClocksThrottleReasonHwSlowdown), ("hw_thermal_slowdown", nv.nvmlClocksThrottleReasonHwThermalSlowdown),
                 ("sw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwThermalSlowdown), ("sw_power_cap", nv.nvmlClocksThrottleReasonSwPowerCap))
        self.source = "nvml"
        while not self.stop_flag:
            self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            for name, bit in names:
                if r & bit:
                    self.reasons.add(name)
            time.sleep(0.005)

    def _run_smi(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                s = [x.strip() for x in out.split(",")] if out else []
                if len(s) >= 8:
                    if s[1].replace(".", "").isdigit():
                        self.sm.append(float(s[1]))
                    if s[2].replace(".", "").isdigit():
                        self.mx.append(float(s[2]))
                    for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[4:8]):
                        if v.lower().startswith("active"):
                            self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.1)

    def run(self):
        try:
            self._run_nvml()
        except Exception:
            self._run_smi()

    def summary(self):
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                "reasons": sorted(self.reasons), "samples": len(self.sm), "source": self.source}


# --------------------------------------------------------------------------------------------------------------
# CPU baseline: the oracle port of the reference's vc() on the host cores (bounded sample of the same workload)
# --------------------------------------------------------------------------------------------------------------
_G = {}
CPU_WHAT = {"reference": "the reference's own vc_wrapper() (oracle/_ref = /root/reference/smCounter.py via oracle/ref_build.py; pysam stand-in over "
                         "in-memory reads, plain dict/set containers)",
            "port": "oracle/smcounter_oracle.py (Python-3 port; oracle/_ref not built)"}


def cpu_kind():
    """'reference': oracle/_ref (the reference's own smCounter.py made runnable by oracle/ref_build.py, plain containers,
    pysam stand-in) is present; 'port': only the oracle restatement is."""
    from oracle import ref_build
    return "reference" if ref_build.available() else "port"


def _cpu_worker(job):
    from oracle import smcounter_oracle as orc
    chrom, pos = job
    p = _G["prm"]
    if _G.get("ref") is not None:          # the reference's vc_wrapper(), exactly as its Pool calls it (smCounter.py:684)
        return _G["ref"].vc_wrapper("bench.bam", chrom, pos, p.minBQ, p.minMQ, p.mtDepth, p.rpb, p.hpLen, p.mismatchThr, p.mtDrop,
                                    p.maxMT, p.primerDist, "bench.fa")
    return orc.vc(_G["index"], chrom, pos, p.minBQ, p.minMQ, p.mtDepth, p.rpb, p.hpLen, p.mismatchThr, p.mtDrop, p.maxMT,
                  p.primerDist, _G["refs"])


def cpu_sample_setup(soa, refs, loci, n_loci_sample, args=None):
    """Pick consecutive loci from the middle of the batch and the reads that overlap them (host objects for the oracle)."""
    import numpy as np
    from oracle import smcounter_oracle as orc
    from smcounter_b200.soa import soa_to_records
    n_loci_sample = max(1, min(int(n_loci_sample), loci.n))
    a = max(0, loci.n // 2 - n_loci_sample // 2)
    sel = np.arange(a, min(loci.n, a + n_loci_sample))
    ends = soa.ref_end()
    mask = np.zeros(soa.n, dtype=bool)
    for rid in np.unique(loci.ref_id[sel]):
        p = loci.pos0[sel[loci.ref_id[sel] == rid]]
        # one window per run of nearby loci (an interval), so that reads between distant intervals are not dragged in
        cuts = np.flatnonzero(np.diff(p) > 1000)
        for lo_i, hi_i in zip(np.concatenate(([0], cuts + 1)), np.concatenate((cuts, [len(p) - 1]))):
            lo, hi = int(p[lo_i]), int(p[hi_i]) + 1
            mask |= (soa.ref_id == rid) & (soa.pos < hi) & (ends > lo)
    recs = soa_to_records(soa.select(np.flatnonzero(mask)), orc.Read)
    _G["index"] = orc.ReadIndex(recs)
    _G["refs"] = refs
    _G["prm"] = vc_params(args)
    _G["ref"] = None
    if cpu_kind() == "reference":
        from oracle import ref_build, ref_shims
        _G["ref"] = ref_build.load("native", inline_pool=False)
        ref_shims.register_bam("bench.bam", _G["index"])
        ref_shims.register_fasta("bench.fa", refs)
    jobs = [(soa.chroms[int(loci.ref_id[i])], str(int(loci.pos0[i]) + 1)) for i in sel]
    return jobs, len(recs)


def cpu_run(jobs, cores, pool=None):
    """loci/s of the oracle port over ``jobs`` on ``cores`` worker processes (the reference's Pool(nCPU) fan-out,
    smCounter.py:683-685); the pool is created and warmed outside the timed region."""
    import multiprocessing as mp
    own = None
    if cores > 1 and pool is None:
        own = pool = mp.get_context("fork").Pool(cores)
        pool.map(_cpu_worker, jobs[:cores], chunksize=1)
    t0 = time.perf_counter()
    if cores > 1:
        rows = pool.map(_cpu_worker, jobs, chunksize=1)
    else:
        rows = [_cpu_worker(j) for j in jobs]
    dt = time.perf_counter() - t0
    if own is not None:
        own.close(); own.join()
    events = sum(int(r.split("\t")[5]) for r in rows if r.split("\t")[5])
    return len(jobs) / dt, dt, events


def pipeline_leg(args, mine, soa, refs, device):
    """The whole reference-facing path, stage by stage, on the first ``--pipeline-intervals`` intervals of the rank-0 batch: BAM
    file -> libsmc_bamio decode -> SoA -> smc_call_batch -> native output stage (rows, repeat filters, called variants) -> the
    three output files (what smCounter.main() does, smCounter.py:645-909).  north_star asks for the end-to-end figure including the
    BAM decode beside the kernel-only one.  One warm-up pass, then ``--pipeline-repeats`` timed passes (median); the BAM itself is
    written outside the timed stages."""
    import shutil
    import tempfile
    from smcounter_b200 import bam, repeats, writers
    from smcounter_b200.rows import headerAll, headerVariants
    from smcounter_b200.shard import reads_for_intervals
    from smcounter_b200.smCounter import call_loci_text
    ivs = mine[:args.pipeline_intervals]
    sub = soa.select(reads_for_intervals(soa, ivs, soa.chroms))
    tmp = tempfile.mkdtemp(prefix="smc_pipe_")
    prm = vc_params(args)
    try:
        path = os.path.join(tmp, "reads.bam")
        bam.write_bam(path, sub, refs.lengths)
        target_rows = [(c, str(s), str(e)) for (c, s, e) in ivs]
        n_loci = sum(e - s for (_, s, e) in ivs)
        runs = []
        reads = None
        for rep in range(1 + max(1, args.pipeline_repeats)):
            reads = None                    # a CLI run decodes once: the previous pass's buffers are released outside the timed stages
            t = [time.perf_counter()]
            reads = bam.read_bam(path, ivs, threads=os.cpu_count() or 1, trim=True)
            t.append(time.perf_counter())
            trf, rm = repeats.build_repeat_regions(target_rows, [], [])
            thr = writers.pi_threshold(prm.mtDepth, 0)
            a, c, v = call_loci_text(reads, ivs, refs, prm, thr, trf, rm, gpus=1, devices=[device], stage_times=(st := {}))
            t.append(time.perf_counter())
            with open(os.path.join(tmp, "out.smCounter.all.txt"), "wb") as fh:
                fh.write(("\t".join(headerAll) + "\n").encode()); fh.write(a)
            with open(os.path.join(tmp, "out.smCounter.cut.txt"), "wb") as fh:
                fh.write(("\t".join(headerVariants) + "\n").encode()); fh.write(c)
            with open(os.path.join(tmp, "out.smCounter.cut.vcf"), "wb") as fh:
                fh.write(writers.vcf_header("out").encode()); fh.write(v)
            t.append(time.perf_counter())
            if rep > 0:
                runs.append((t[3] - t[0], t[1] - t[0], t[2] - t[1], t[3] - t[2], dict(st), int(reads.n)))
        if os.environ.get("SMC_PROFILE_PIPELINE"):          # where the host time of one pass goes (stderr)
            import cProfile
            import pstats
            pr = cProfile.Profile()
            pr.enable()
            reads = bam.read_bam(path, ivs, threads=os.cpu_count() or 1, trim=True)
            call_loci_text(reads, ivs, refs, prm, thr, trf, rm, gpus=1, devices=[device])
            pr.disable()
            pstats.Stats(pr, stream=sys.stderr).sort_stats("tottime").print_stats(25)
        runs.sort(key=lambda r: r[0])
        tot, dec, call, wr, st, nreads = runs[len(runs) // 2]
        return {"value": n_loci / tot, "unit": UNIT, "loci": n_loci, "reads": nreads, "intervals": len(ivs), "repeats": len(runs), "warmup": 1,
                "bam_mb": os.path.getsize(path) / 1e6, "ms_total": 1e3 * tot, "ms_bam_decode": 1e3 * dec, "ms_call_loci_text": 1e3 * call,
                "ms_gpu_call": st.get("ms_gpu_call"), "ms_rows_filters_calls_native": st.get("ms_format_rows"), "ms_write_files": 1e3 * wr,
                "gpu_call_detail": {k: v for k, v in st.items() if k not in ("ms_gpu_call", "ms_format_rows")},
                "all_runs_ms": [round(1e3 * r[0], 2) for r in runs],
                "what": "median of %d passes after 1 warm-up: BAM decode (libsmc_bamio, all host threads, trimmed on the fly) + context + smc_call_batch + "
                        "device HP/LowC + native rows / repeat filters / called-variant lines (libsmc_bamio: smc_rows_emit) + the three files" % len(runs)}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def strong_leg(args, ivs, soa, refs, n_gpus):
    """Strong scaling of the product path: ONE fixed panel (the rank-0 batch 0: its intervals and all their reads, trimmed
    as the BAM decoder delivers them) through ``smCounter.call_loci(gpus=N)`` from ONE process -- the drop-in for the
    reference's Pool fan-out (smCounter.py:683-685): shards by BED interval, one host thread and up to three contexts per GPU,
    rows formatted by the native output stage.  Median of 5 calls after one warm-up."""
    from smcounter_b200.smCounter import call_loci
    prm = vc_params(args)
    reads = soa.trim_to_targets(ivs)
    n_loci = sum(e - s for (_, s, e) in ivs)
    runs = []
    for rep in range(6):
        t0 = time.perf_counter()
        rows = call_loci(reads, ivs, refs, prm, gpus=n_gpus, devices=list(range(n_gpus)), stage_times=(st := {}))
        dt = time.perf_counter() - t0
        assert len(rows) == n_loci
        if rep:
            runs.append((dt, dict(st)))
    if os.environ.get("SMC_PROFILE_STRONG"):            # where the host time of one call goes (stderr)
        import cProfile
        import pstats
        pr = cProfile.Profile()
        pr.enable()
        call_loci(reads, ivs, refs, prm, gpus=n_gpus, devices=list(range(n_gpus)))
        pr.disable()
        pstats.Stats(pr, stream=sys.stderr).sort_stats("cumulative").print_stats(35)
    runs.sort(key=lambda r: r[0])
    dt, st = runs[len(runs) // 2]
    return {"value": n_loci / dt, "unit": UNIT, "gpus": n_gpus, "loci": n_loci, "reads": int(reads.n), "intervals": len(ivs), "ms": 1e3 * dt,
            "all_runs_ms": [round(1e3 * r[0], 2) for r in runs], "ms_plan": st.get("ms_plan"), "ms_select_pack_sum": st.get("ms_select_pack"), "ms_ctx_create_sum": st.get("ms_ctx_create"),
            "ms_gpu_call_sum": st.get("ms_gpu_call"), "ms_format_rows_sum": st.get("ms_format_rows"),
            "batches": st.get("batches"),
            "what": "smCounter.call_loci(reads, intervals, gpus=%d) on one fixed panel from one process (plan_shards by BED interval, one thread and "
                    "up to three contexts per GPU, each batch packed natively into pinned buffers, rows through smc_rows_emit); total work fixed as N grows" % n_gpus}


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cores = os.cpu_count() or 1

    if args.impl == "reference":
        # The reference arm: the reference's own per-locus code (oracle/_ref: /root/reference/smCounter.py made runnable by
        # oracle/ref_build.py; the oracle port if that is not built) behind a multiprocessing.Pool over all host cores, exactly as
        # smCounter.py:683-685 fans it out.  Rank 0 only.  Same workload and config as the CUDA arm; each step is a bounded
        # sample of it (consecutive loci of the first batch), sized so that the run ends within minutes.
        if rank != 0:
            return 0
        ivs0, _, refs, loci, bed_order, soa = make_batches(args, 0, 1, only_first=True)[0]
        n_sample = args.cpu_loci or 16 * cores
        jobs, nrec = cpu_sample_setup(soa, refs, loci, n_sample, args)
        import multiprocessing as mp
        pool = mp.get_context("fork").Pool(cores) if cores > 1 else None
        for _ in range(min(args.warmup, 1)):
            cpu_run(jobs[:max(1, 2 * cores)], cores, pool)
        times, ev = [], 0
        for _ in range(args.steps):
            v, dt, ev = cpu_run(jobs, cores, pool)
            times.append(dt)
        if pool is not None:
            pool.close(); pool.join()
        value = len(jobs) * len(times) / sum(times)
        sample = "%d consecutive loci of batch 0 per step (%d reads, %d pileup events) x %d steps; %s; multiprocessing.Pool(%d)" % (
            len(jobs), nrec, ev, args.steps, CPU_WHAT[cpu_kind()], cores)
        line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1000.0 * sum(times) / len(times), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "int32+f64", "data": "synthetic", "config": config_dict(args, max(1, args.gpus)),
                "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": cpu_kind(), "sample": sample},
                "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    import numpy as np
    import torch
    import torch.distributed as dist
    from smcounter_b200.caller import GpuCaller, LocusResults
    from smcounter_b200.rows import device_hp_flags

    torch.cuda.set_device(local_rank)
    all_cpus = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    numa = None
    if world > 1 and all_cpus is not None:
        # one process per GPU: run on the cores next to this GPU so that the pinned host buffers (first touch) live on its
        # NUMA node and the uploads of the 8 ranks do not all cross the socket interconnect
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(local_rank)
            words = nv.nvmlDeviceGetCpuAffinity(h, (max(all_cpus) + 64) // 64)
            local = {64 * w + b for w, x in enumerate(words) for b in range(64) if (int(x) >> b) & 1} & set(all_cpus)
            if local:
                os.sched_setaffinity(0, local)
                numa = len(local)
        except Exception:
            numa = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        host_group = dist.new_group(backend="gloo")          # waits that must not park a kernel on the GPU
    batches = make_batches(args, rank, world)
    prm = vc_params(args)
    NB = len(batches)

    # pinned host copies of every buffer that crosses the ABI
    def pin(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        return t.numpy()
    for (_, soa, _, loci, _, _) in batches:
        for f in ("ref_id", "pos", "flag", "mapq", "nm", "l_seq", "n_cigar", "umi", "frag_id", "seq", "qual", "cigar"):
            setattr(soa, f, pin(getattr(soa, f)))
        if not soa.packed:
            for f in ("seq_off", "qual_off", "cigar_off"):
                setattr(soa, f, pin(getattr(soa, f)))
        for f in ("store_lo", "store_len", "qual_lut"):
            if getattr(soa, f) is not None:
                setattr(soa, f, pin(getattr(soa, f)))
        if soa.seq_exc is not None:
            soa.seq_exc = tuple(pin(a) for a in soa.seq_exc)
        for f in ("ref_id", "pos0", "ref_base"):
            setattr(loci, f, pin(getattr(loci, f)))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- kernel-only: every batch resident in HBM (one context per batch)
    res_callers = []
    for (_, soa, _, loci, _, _) in batches:
        c = GpuCaller(prm, device=local_rank)
        c.upload(soa, loci)
        res_callers.append(c)
    for _ in range(args.warmup):
        for c in res_callers:
            c.run()
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    t0 = time.perf_counter()
    dev_ms, launches = 0.0, 0
    stage = {}
    tms0 = None
    for _ in range(args.steps):
        for k, c in enumerate(res_callers):
            c.run()
            tm = c.timings()
            dev_ms += tm["ms_total_device"]; launches += tm["kernel_launches"]
            for key in ("ms_prep", "ms_sort", "ms_pileup", "ms_stats", "ms_k_pileup", "ms_k_gather", "ms_k_merge", "ms_read_sort", "ms_k_read_prep", "ms_event_sort"):
                stage[key] = stage.get(key, 0.0) + tm[key]
            if k == 0:
                tms0 = tm
    barrier()
    wall_s = time.perf_counter() - t0
    events_rank = reads_rank = tile_events_rank = 0
    prep_bytes = 0
    outs = []
    for c, (_, soa, _, loci, _, _) in zip(res_callers, batches):
        tm = c.timings()
        events_rank += int(tm["n_pileup_events"]); reads_rank += int(tm["n_reads"]); tile_events_rank += int(tm["n_tile_events"])
        prep_bytes += int(tm["read_prep_bytes"])
        outs.append(c.download(LocusResults(loci.n, max(int(tm["n_dyn"]), 16), pinned=True)))
        c.close()
    n_dyn = sum(o.n_dyn for o in outs)
    if args.dump_outputs:           # before the end-to-end leg reuses these buffers
        dump_outputs(args.dump_outputs, outs, prefix="rank%d." % rank if world > 1 else "", share=world)

    # ---------------- end to end: host buffers in, host buffers out, every step: smc_call_batch (pipelined upload, kernels,
    # download) and the device HP / LowC pass over the candidates of the batch (smc_hp_lowcomp)
    # As smCounter._run_shards does: three contexts and three host threads per GPU, so that one batch uploads while the previous ones
    # computes and downloads (ctypes drops the GIL inside the library).
    import queue
    from concurrent.futures import ThreadPoolExecutor
    n_ctx = min(int(os.environ.get("SMC_CTX_PER_GPU", "3")), NB)
    callers = [GpuCaller(prm, device=local_rank) for _ in range(n_ctx)]
    free = queue.SimpleQueue()
    for i in range(n_ctx):
        free.put(i)
    pool = ThreadPoolExecutor(max_workers=n_ctx)

    host_tl = [] if os.environ.get("SMC_TIMELINE") else None      # debugging: host-side stamps of every e2e batch

    def e2e_batch(k):
        (_, soa, refs, loci, _, _), out = batches[k], outs[k]
        t_a = time.perf_counter()
        i = free.get()
        try:
            t_b = time.perf_counter()
            res = callers[i].call(soa, loci, out=out)
            t_c = time.perf_counter()
            tm = callers[i].timings()
            device_hp_flags(callers[i], res, soa, loci, soa.chroms, refs, prm.hpLen)
            if host_tl is not None:
                host_tl.append((k, i, t_a, t_b, t_c, time.perf_counter()))
            return tm
        finally:
            free.put(i)

    def e2e_pass(steps):
        # the batches of all the steps go through the contexts as one stream, the way a long job's shards do
        # (smCounter._run_shards): no barrier between steps, so a batch uploads while the one before it computes
        tms = list(pool.map(e2e_batch, [k % NB for k in range(steps * NB)]))
        last = tms[-NB:]
        return sum(int(t["bytes_h2d"]) for t in last), sum(int(t["bytes_d2h"]) for t in last), tms[-1]
    # warm-up: every context meets every batch once (its device buffers grow to the largest one), then the streamed passes
    for i in range(len(callers)):
        for k in range(NB):
            callers[i].call(batches[k][1], batches[k][3], out=outs[k])
    if args.warmup:
        e2e_pass(min(args.warmup, 2))
    barrier()
    t1 = time.perf_counter()
    h2d_b, d2h_b, e2e_tm = e2e_pass(args.steps)
    e2e_s_own = time.perf_counter() - t1          # this rank alone (the straggler table); the headline waits for everybody
    barrier()
    e2e_s = time.perf_counter() - t1
    if host_tl:
        for (k, i, t_a, t_b, t_c, t_d) in host_tl[-3 * NB:]:
            print("[bench timeline] batch %d ctx %d: task %.2f got ctx %.2f call done %.2f hp flags done %.2f (ms since the timed region began)"
                  % (k, i, 1e3 * (t_a - t1), 1e3 * (t_b - t1), 1e3 * (t_c - t1), 1e3 * (t_d - t1)), file=sys.stderr)
    sampler.stop_flag = True
    sampler.join(timeout=2)
    pool.shutdown(wait=True)
    for c in callers:
        c.close()

    def allred(x, op):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=op)
        return float(t.item())
    allmax = lambda x: allred(x, dist.ReduceOp.MAX)
    allsum = lambda x: allred(x, dist.ReduceOp.SUM)

    loci_rank = float(sum(b[3].n for b in batches))
    dev_s_max = allmax(dev_ms / 1000.0)
    wall_s_max = allmax(wall_s)
    e2e_s_max = allmax(e2e_s)
    e2e_s_min = -allmax(-e2e_s_own)
    loci_total = allsum(loci_rank)
    # who is the straggler: every rank's own e2e / device time per step and the H2D of its last batch
    mine_stats = [float(rank), 1000.0 * e2e_s_own / args.steps, 1000.0 * (dev_ms / 1000.0) / args.steps, float(e2e_tm["ms_h2d"]),
                  float(e2e_tm["bytes_h2d"]) / float(e2e_tm["ms_h2d"]) / 1e6 if e2e_tm["ms_h2d"] > 0 else 0.0, float(e2e_tm["ms_total_device"])]
    if world > 1:
        tl = [torch.zeros(len(mine_stats), dtype=torch.float64, device="cuda") for _ in range(world)]
        dist.all_gather(tl, torch.tensor(mine_stats, dtype=torch.float64, device="cuda"))
        all_stats = [t.tolist() for t in tl]
    else:
        all_stats = [mine_stats]
    per_rank = [{"rank": int(a[0]), "e2e_ms_per_step": a[1], "resident_ms_per_step": a[2], "last_batch_ms_h2d": a[3], "last_batch_h2d_gbs": a[4],
                 "last_batch_ms_device": a[5]} for a in all_stats]
    events_total = allsum(float(events_rank))
    reads_total = allsum(float(reads_rank))
    # device time is what the CUDA events on the library's launch stream bracket for each batch run (it contains the host
    # round-trips a run needs); wall clock is reported beside it.
    value = loci_total * args.steps / dev_s_max
    e2e_value = loci_total * args.steps / e2e_s_max

    line = None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        nrun = args.steps * NB                                   # batch runs in the timed region of this rank
        algo_bytes = ALGO_BYTES_PER_EVENT * float(events_rank) / NB          # per launch pair (one batch), averaged over the rank's batches
        kp_avg_s = stage["ms_k_pileup"] / nrun / 1000.0
        traffic = None          # dram__bytes_read.sum + dram__bytes_write.sum of one k_gather + k_merge launch pair (ncu --set full, batch 0)
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "k_pileup_traffic.json")))
            if int(tr["pileup_events"]) == int(tms0["n_pileup_events"]):
                traffic = int(tr["dram_bytes_read"]) + int(tr["dram_bytes_write"])
        except Exception:
            pass
        achieved = algo_bytes / kp_avg_s / 1e9 if kp_avg_s > 0 else 0.0
        step_s = (dev_ms / nrun) / 1000.0
        soa0 = batches[0][1]
        gbs = lambda b, ms: (b / (ms / 1000.0) / 1e9) if ms > 0 else None
        n_r, n_te = reads_rank / NB, tile_events_rank / NB
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": 1000.0 * dev_s_max / args.steps, "wall_ms_per_step": 1000.0 * wall_s_max / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32+f64", "data": "synthetic",
                "config": config_dict(args, world),
                "workload_stats": {"loci_total": int(loci_total), "reads_total": int(reads_total), "pileup_events_per_step": int(events_total),
                                   "tile_events_per_step_rank0": int(tile_events_rank), "pileup_events_batch0_rank0": int(tms0["n_pileup_events"]), "resident_mb_rank0": sum(b[1].nbytes() for b in batches) / 1e6,
                                   "reads": "whole reads" if soa0.store_lo is None else "bases / qualities trimmed to each read's target window (store_lo / store_len), "
                                            "%.0f of %d bases per read stored" % (float(soa0.store_len.mean()), int(soa0.l_seq.max())) +
                                            ("; compact upload: %d-bit scalars, %d-bit quality codes, %d-bit bases" % (soa0.scalar_bits, soa0.qual_bits, soa0.seq_bits)
                                             if soa0.scalar_bits != 32 or soa0.qual_bits != 8 else ""),
                                   "host_affinity": ("GPU-local cores (%d) while pinning and uploading" % numa) if numa else "unbound"},
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d_b), "d2h_bytes_per_step": int(d2h_b),
                        "ms_per_step": 1000.0 * e2e_s_max / args.steps, "ms_per_step_fastest_rank": 1000.0 * e2e_s_min / args.steps,
                        "last_batch": {"ms_h2d": e2e_tm["ms_h2d"], "ms_device": e2e_tm["ms_total_device"], "ms_d2h": e2e_tm["ms_d2h"],
                                       "h2d_gbs": e2e_tm["bytes_h2d"] / e2e_tm["ms_h2d"] / 1e6 if e2e_tm["ms_h2d"] > 0 else None},
                        "what": "per step and GPU: %d x (smc_call_batch from pinned host buffers -- scalars first, bases / qualities in %d chunks on a copy "
                                "stream, %d pileup launch pairs as they arrive -- + download + smc_hp_lowcomp over the batch's candidates); %d contexts / host threads per GPU taking turns on the link, so the next batch uploads while the previous ones compute and download"
                                % (NB, e2e_tm["pipe_chunks"], e2e_tm["pipe_launches"], n_ctx)},
                "per_rank": per_rank,
                "gpu_launches": int(launches),
                "stage_ms_per_batch_rank0": {k: v / nrun for k, v in stage.items()},
                "roofline": {"bound": "hbm", "limited_by": "instruction issue (ncu, profiles/r02_k_gather_*_summary.txt: issue slots 70 % busy, DRAM 6 %): the tile "
                                                          "design never materialises the per-(read, locus) events the 35 B / event figure charges for",
                             "kernel": "k_gather + k_merge (K3: tile pileup = event expansion + fragment merge, then calProb / PI / consensus)",
                             "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None,
                             "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
                             "algorithmic_bytes_per_launch": algo_bytes, "bytes_per_event": ALGO_BYTES_PER_EVENT,
                             "ms_per_launch": 1000.0 * kp_avg_s, "traffic": traffic,
                             "whole_step": {"what": "the same 35 B x pileup events over the WHOLE device run of a batch (read sort, prep, tile events, "
                                                    "both pileup kernels, ALT / filters / Fisher), rank 0",
                                            "achieved": algo_bytes / step_s / 1e9 if step_s > 0 else 0.0,
                                            "frac": algo_bytes / step_s / 1e9 / peak if step_s > 0 and peak else None},
                             "other_kernels": {
                                 "k_read_prep": {"ms": stage["ms_k_read_prep"] / nrun, "algorithmic_bytes": prep_bytes / NB,
                                                 "achieved_gbs": gbs(prep_bytes / NB, stage["ms_k_read_prep"] / nrun)},
                                 "read_sort": {"ms": stage["ms_read_sort"] / nrun, "passes": int(tms0["read_sort_passes"]),
                                               "algorithmic_bytes": 24.0 * n_r * int(tms0["read_sort_passes"]),
                                               "achieved_gbs": gbs(24.0 * n_r * int(tms0["read_sort_passes"]), stage["ms_read_sort"] / nrun),
                                               "what": "per pass 12 B read + 12 B written per read (u64 key + u32 index); histogram, scan and scatter kernels"},
                                 "tile_event_sort": {"ms": stage["ms_event_sort"] / nrun, "algorithmic_bytes": 24.0 * n_te,
                                                     "achieved_gbs": gbs(24.0 * n_te, stage["ms_event_sort"] / nrun)}},
                             "events_per_s": float(events_rank) / NB / kp_avg_s if kp_avg_s > 0 else 0.0},
                "clocks": sampler.summary(), "n_dyn_alleles_rank0": int(n_dyn), "n_fisher_rank0": int(tms0["n_fisher"])}

    if all_cpus is not None and numa:
        os.sched_setaffinity(0, all_cpus)          # the host-side legs below may use every core again
    ivs0, _, refs0, loci0, _, full0 = batches[0]
    if rank == 0 and args.pipeline_intervals > 0 and full0 is not None:
        try:
            line["pipeline"] = pipeline_leg(args, ivs0, full0, refs0, local_rank)
        except Exception as e:          # the extra leg must never cost the bench line
            line["pipeline"] = {"error": repr(e)}

    if world > 1:
        dist.barrier()                      # every rank has finished its timed legs and closed its contexts: the GPUs are idle
    if rank == 0 and not args.no_strong and full0 is not None:
        try:
            line["strong"] = strong_leg(args, ivs0, full0, refs0, world)
        except Exception as e:
            line["strong"] = {"error": repr(e)}

    if rank == 0 and not args.no_cpu_baseline and full0 is not None:
        n_sample = args.cpu_loci or 24 * cores          # ~10-30 s of host work
        jobs, nrec = cpu_sample_setup(full0, refs0, loci0, n_sample, args)
        v, dt, ev = cpu_run(jobs, cores)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": cpu_kind(),
                                "sample": "%d consecutive loci of the rank-0 batch 0 (%d reads, %d pileup events), %s "
                                          "with multiprocessing.Pool(%d), %.1f s" % (len(jobs), nrec, ev, CPU_WHAT[cpu_kind()], cores, dt),
                                "archived_reference": "4.15 loci/s on 10 processes at DP~58k (example run log, 2017 hardware)"}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.barrier(group=host_group)
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
