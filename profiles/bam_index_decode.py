"""Decode time and memory of read_bam with and without the BAM index, for target BEDs that cover 100 %, 10 % and 1 % of a
panel's intervals.

One indexed BAM of the N0030 panel geometry (bench.py's cfg2 read model, fixed seed) is written to a temporary directory.  For
every BED (every k-th interval, k = 1, 10, 100) and each path -- indexed (the .bai beside the BAM) and whole file (a link to the
same BAM without one) -- a fresh subprocess runs read_bam(..., trim=True) once as a warm-up and five times timed, and reports
the median wall time, the growth of its peak RSS (VmHWM) during the decode, the reads kept, and the compressed bytes read and
bytes inflated (the decoder's SMC_BAM_TIMING lines).  One JSON line per BED on stdout.

    python profiles/bam_index_decode.py [--intervals 100] [--seed 1] [--out FILE]
"""
import argparse
import json
import os
import platform
import re
import shutil
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
SPEC = dict(umis_per_locus=3000, rpb=4.0, snv_every=1000, snv_vaf=0.01, indel_every=12000, indel_vaf=0.01)     # bench.py cfg2


def _hwm_kb():
    with open("/proc/self/status") as fh:
        return int(re.search(r"VmHWM:\s+(\d+)", fh.read()).group(1))


def child(path, bed, repeats):
    """One case in this process: prints one JSON object."""
    from smcounter_b200 import bam
    from smcounter_b200.synth import panel_intervals_from_bed
    ivs = panel_intervals_from_bed(bed)
    threads = os.cpu_count() or 1
    base = _hwm_kb()
    reads = bam.read_bam(path, ivs, threads=threads, trim=True)                  # warm-up (page cache, thread start-up)
    n = reads.n
    rss = (_hwm_kb() - base) / 1024.0
    del reads
    times = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        r = bam.read_bam(path, ivs, threads=threads, trim=True)
        times.append(1e3 * (time.perf_counter() - t0))
        assert r.n == n
        del r
    # byte counts from the decoder's own timing lines, on one more decode with fd 2 sent to a file
    os.environ["SMC_BAM_TIMING"] = "1"
    log = tempfile.TemporaryFile(mode="w+")
    saved = os.dup(2)
    os.dup2(log.fileno(), 2)
    try:
        bam.read_bam(path, ivs, threads=threads, trim=True)
    finally:
        os.dup2(saved, 2)
        os.close(saved)
    log.seek(0)
    comp = infl = 0
    for m in re.finditer(r"compressed bytes read (\d+), inflated bytes (\d+)", log.read()):
        comp += int(m.group(1)); infl += int(m.group(2))
    print(json.dumps(dict(median_ms=round(statistics.median(times), 2), times_ms=[round(t, 2) for t in times], peak_rss_growth_mb=round(rss, 1),
                          reads=int(n), compressed_bytes_read=comp, inflated_bytes=infl, index_used=bam.find_index(path) is not None)))


def cpu_model():
    try:
        with open("/proc/cpuinfo") as fh:
            m = re.search(r"model name\s*:\s*(.*)", fh.read())
            return m.group(1).strip() if m else platform.processor()
    except OSError:
        return platform.processor()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--intervals", type=int, default=100, help="panel intervals in the BAM (seeded subset of the N0030 BED)")
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--child", nargs=2, metavar=("BAM", "BED"), help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.child:
        return child(a.child[0], a.child[1], a.repeats)
    from smcounter_b200 import bam
    from smcounter_b200.synth import SynthSpec, make_panel_mp, panel_intervals_from_bed
    ivs = panel_intervals_from_bed(os.path.join(ROOT, "tests", "golden", "n0030_panel.bed"), limit=a.intervals, seed=a.seed)
    tmp = tempfile.mkdtemp(prefix="smc_bai_")
    lines = []
    try:
        t0 = time.perf_counter()
        soa, refs, _ = make_panel_mp(ivs, SynthSpec(**SPEC), seed=a.seed, n_groups=16)
        path = os.path.join(tmp, "reads.bam")
        bam.write_bam(path, soa, refs.lengths, index=True)
        whole = os.path.join(tmp, "whole.bam")                   # the same file without an index beside it
        os.symlink(path, whole)
        head = dict(what="bam_index_decode setup", host_cpu=cpu_model(), host_cores=os.cpu_count(), intervals=len(ivs), reads_in_bam=int(soa.n),
                    bam_bytes=os.path.getsize(path), bai_bytes=os.path.getsize(path + ".bai"), setup_s=round(time.perf_counter() - t0, 1))
        del soa
        lines.append(head)
        print(json.dumps(head), flush=True)
        for k, label in ((1, "100%"), (10, "10%"), (100, "1%")):
            bed = os.path.join(tmp, "k%d.bed" % k)
            sub = ivs[::k]
            with open(bed, "w") as fh:
                fh.write("".join("%s\t%d\t%d\n" % iv for iv in sub))
            res = {}
            for mode, p in (("indexed", path), ("whole_file", whole)):
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", p, bed, "--repeats", str(a.repeats)],
                                   capture_output=True, text=True, check=True)
                res[mode] = json.loads(r.stdout.strip().splitlines()[-1])
            assert res["indexed"]["index_used"] and not res["whole_file"]["index_used"]
            assert res["indexed"]["reads"] == res["whole_file"]["reads"]
            line = dict(what="bam_index_decode", bed=label, every_kth=k, bed_intervals=len(sub), **res,
                        time_whole_over_indexed=round(res["whole_file"]["median_ms"] / res["indexed"]["median_ms"], 2),
                        rss_whole_over_indexed=round(res["whole_file"]["peak_rss_growth_mb"] / max(res["indexed"]["peak_rss_growth_mb"], 0.1), 2))
            lines.append(line)
            print(json.dumps(line), flush=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    if a.out:
        with open(a.out, "a") as fh:
            fh.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
