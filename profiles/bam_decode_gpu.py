"""Decode time of read_bam on the host and on the GPU (--bamDecoder gpu: smc_decode_bam), for target BEDs that cover 100 %,
10 % and 1 % of a panel's intervals, through the BAM index and from the whole file.

One indexed BAM of the N0030 panel geometry (bench.py's cfg2 read model, fixed seed) is written to a temporary directory, as in
profiles/bam_index_decode.py.  For every BED, path (indexed / whole file) and decoder, a fresh subprocess runs
read_bam(..., trim=True) once as a warm-up and five times timed, and reports the median wall time, the reads kept and, for the
GPU, the per-stage CUDA-event times of one more decode (SMC_BAM_TIMING lines).  Both decoders' arrays are checked equal.  One
JSON line per (BED, path) on stdout, the GPU's name and power limit in the setup line.

--variant-lib LIB also times the GPU decode with another build of libsmc_b200 (e.g. one compiled with
-DSMC_INFLATE_LOCAL_TABLES: the inflate tables in local memory instead of shared memory) beside the default one.

--pipeline: instead, the stages of smCounter.main() on bench.py's 96-interval batch -- bench.py's own pipeline leg (BAM decode,
smc_call_batch, rows / filters / called variants, the three files; median of 5 passes after a warm-up) -- once with each
decoder, one process each; one JSON line per decoder.

    python profiles/bam_decode_gpu.py [--intervals 100] [--seed 1] [--variant-lib LIB] [--out FILE]
    python profiles/bam_decode_gpu.py --pipeline [--out FILE]
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


def child(path, bed, repeats, decoder):
    """One case in this process: prints one JSON object."""
    import numpy as np
    from smcounter_b200 import bam
    from smcounter_b200.synth import panel_intervals_from_bed
    ivs = panel_intervals_from_bed(bed)
    threads = os.cpu_count() or 1
    dev = 0 if decoder == "gpu" else None
    reads = bam.read_bam(path, ivs, threads=threads, trim=True, device=dev)      # warm-up (page cache, threads, CUDA context)
    n = reads.n
    digest = [int(np.bitwise_xor.reduce(np.frombuffer(getattr(reads, f).tobytes(), np.uint8).astype(np.uint64) *
                                        (1 + np.arange(getattr(reads, f).nbytes, dtype=np.uint64)))) for f in ("frag_id", "umi", "qual", "seq", "store_lo")]
    assert reads.__dict__.get("_bam_decoder") == ("device" if dev is not None else "host")
    del reads
    times = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        r = bam.read_bam(path, ivs, threads=threads, trim=True, device=dev)
        times.append(1e3 * (time.perf_counter() - t0))
        assert r.n == n
        del r
    stages = {}
    if dev is not None:                  # per-stage device times from the decoder's own timing lines, one more decode
        os.environ["SMC_BAM_TIMING"] = "1"
        log = tempfile.TemporaryFile(mode="w+")
        saved = os.dup(2)
        os.dup2(log.fileno(), 2)
        try:
            bam.read_bam(path, ivs, threads=threads, trim=True, device=dev)
        finally:
            os.dup2(saved, 2)
            os.close(saved)
        log.seek(0)
        for m in re.finditer(r"\[smc_b200\] bam decode ([^:]+): ([0-9.]+) ms", log.read()):
            stages[m.group(1)] = float(m.group(2))
    print(json.dumps(dict(median_ms=round(statistics.median(times), 2), times_ms=[round(t, 2) for t in times], reads=int(n), digest=digest,
                          device_stage_ms=stages, index_used=bam.find_index(path) is not None)))


def pipeline_child(decoder):
    """bench.py's pipeline leg with read_bam on the host or on GPU 0: prints one JSON object"""
    import functools
    import bench
    from smcounter_b200 import bam
    args = bench.parse_args(["--gpus", "1"])
    ivs0, _, refs0, _, _, full0 = bench.make_batches(args, 0, 1, only_first=True)[0]
    if decoder == "gpu":
        orig = bam.read_bam
        bam.read_bam = functools.partial(orig, device=0)
    res = bench.pipeline_leg(args, ivs0, full0, refs0, 0)
    print(json.dumps(res))


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
    ap.add_argument("--variant-lib", default=None, help="another build of libsmc_b200.so to time the GPU decode with")
    ap.add_argument("--pipeline", action="store_true", help="the stages of main() on bench.py's 96-interval batch, per decoder")
    ap.add_argument("--child", nargs=3, metavar=("BAM", "BED", "DECODER"), help=argparse.SUPPRESS)
    ap.add_argument("--pipeline-child", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.child:
        return child(a.child[0], a.child[1], a.repeats, a.child[2])
    if a.pipeline_child:
        return pipeline_child(a.pipeline_child)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    gpu = gpu.splitlines()[0] if gpu else None
    if a.pipeline:
        lines = []
        for decoder in ("host", "gpu"):
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--pipeline-child", decoder], capture_output=True, text=True,
                               check=True, cwd=ROOT)
            res = json.loads(r.stdout.strip().splitlines()[-1])
            line = dict(what="bam_decode_gpu pipeline (stages of smCounter.main() on bench.py's 96-interval batch)", decoder=decoder, gpu=gpu,
                        host_cpu=cpu_model(), host_cores=os.cpu_count(), pipeline=res)
            lines.append(line)
            print(json.dumps(line), flush=True)
        if a.out:
            with open(a.out, "a") as fh:
                fh.write("".join(json.dumps(x) + "\n" for x in lines))
        return
    from smcounter_b200 import bam
    from smcounter_b200.synth import SynthSpec, make_panel_mp, panel_intervals_from_bed
    ivs = panel_intervals_from_bed(os.path.join(ROOT, "tests", "golden", "n0030_panel.bed"), limit=a.intervals, seed=a.seed)
    tmp = tempfile.mkdtemp(prefix="smc_bamgpu_")
    lines = []
    try:
        t0 = time.perf_counter()
        soa, refs, _ = make_panel_mp(ivs, SynthSpec(**SPEC), seed=a.seed, n_groups=16)
        path = os.path.join(tmp, "reads.bam")
        bam.write_bam(path, soa, refs.lengths, index=True)
        whole = os.path.join(tmp, "whole.bam")                   # the same file without an index beside it
        os.symlink(path, whole)
        head = dict(what="bam_decode_gpu setup", gpu=gpu, variant_lib=a.variant_lib and os.path.basename(a.variant_lib), host_cpu=cpu_model(), host_cores=os.cpu_count(), intervals=len(ivs), reads_in_bam=int(soa.n),
                    bam_bytes=os.path.getsize(path), bai_bytes=os.path.getsize(path + ".bai"), setup_s=round(time.perf_counter() - t0, 1))
        del soa
        lines.append(head)
        print(json.dumps(head), flush=True)
        for k, label in ((1, "100%"), (10, "10%"), (100, "1%")):
            bed = os.path.join(tmp, "k%d.bed" % k)
            sub = ivs[::k]
            with open(bed, "w") as fh:
                fh.write("".join("%s\t%d\t%d\n" % iv for iv in sub))
            for mode, p in (("indexed", path), ("whole_file", whole)):
                res = {}
                for decoder, lib in (("host", None), ("gpu", None)) + ((("gpu_variant", a.variant_lib),) if a.variant_lib else ()):
                    env = dict(os.environ, **({"SMC_B200_LIB": os.path.abspath(lib)} if lib else {}))
                    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", p, bed, "gpu" if lib else decoder, "--repeats",
                                        str(a.repeats)], capture_output=True, text=True, check=True, env=env)
                    res[decoder] = json.loads(r.stdout.strip().splitlines()[-1])
                assert all(res[d]["digest"] == res["host"]["digest"] and res[d]["reads"] == res["host"]["reads"] for d in res)
                line = dict(what="bam_decode_gpu", bed=label, every_kth=k, bed_intervals=len(sub), path=mode, **res,
                            host_over_gpu=round(res["host"]["median_ms"] / res["gpu"]["median_ms"], 2))
                lines.append(line)
                print(json.dumps(line), flush=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    if a.out:
        with open(a.out, "a") as fh:
            fh.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
