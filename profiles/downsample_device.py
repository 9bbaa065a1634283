"""Down-sampling drawn on the device, measured on one GPU: one cfg2 batch of bench.py (96 intervals, trimmed + compact upload).

  A. maxMT = 1000: every covered locus has more barcodes than ds and is drawn.
     - resident run with the device draw (smc_set_downsample(SMC_DS_DEVICE)): ms_total_device (CUDA events, the whole run:
       first pileup + statistics, draw, second pileup + statistics) and the wall time of smc_run_resident;
     - the draw alone: one run under torch.profiler, the device span from the first to the last kernel of the draw (numbering
       of the flagged loci, listing pass, insertion-order sort, hashes, draw, sort of the kept codes, mask CSR) and the kernel
       time summed by name;
     - call_loci wall time for the batch (whole reads in, rows out), which now draws on the device;
     - the host draw of the parent's path (downsample.draw_keep_masks: device listing + Python draw) on a sample of the flagged
       loci, per locus, EXTRAPOLATED to all flagged loci.
  B. maxMT = 0 (the default cfg2, nothing flagged): resident ms_total_device of the parent build (--parent-lib), this build with
     the mode off, and this build with the device draw on, alternating in one process.

Prints one JSON line per result and writes them to --out.  Card name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def emit(out, rec):
    line = json.dumps(rec)
    print(line, flush=True)
    out.write(line + "\n")
    out.flush()


def load_lib(path):
    """A GpuCaller factory bound to this build (path None) or to the library at ``path``, e.g. the parent commit's build, which
    lacks the device-draw entry points: its functions take the signatures this build's binding declares."""
    import ctypes as C
    from smcounter_b200 import _ffi
    from smcounter_b200.caller import GpuCaller
    lib = _ffi.load()
    if path:
        mine, lib = lib, C.CDLL(os.path.abspath(path))
        for name in _ffi.EXPORTS:
            if hasattr(lib, name):
                f, g = getattr(lib, name), getattr(mine, name)
                f.argtypes, f.restype = g.argtypes, g.restype

    def make(prm, **kw):
        saved, _ffi._lib = _ffi._lib, lib
        try:
            return GpuCaller(prm, **kw)
        finally:
            _ffi._lib = saved
    return make


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", default=None, help="libsmc_b200.so of the parent commit for leg B")
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "downsample_device.jsonl"))
    ap.add_argument("--runs", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--host-sample", type=int, default=200)
    a = ap.parse_args()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    out = open(a.out, "w")
    import torch
    import bench
    from smcounter_b200 import _ffi
    from smcounter_b200.caller import UmiKeep
    from smcounter_b200.downsample import draw_keep_masks
    from smcounter_b200.smCounter import call_loci
    torch.cuda.init()
    gpu = card()
    bargs = bench.parse_args(["--batches", "1"])
    ivs, soa, refs, loci, _, full = bench.make_batches(bargs, 0, 1, only_first=True)[0]
    base = dict(gpu=gpu, workload="cfg2 batch 0 (%d intervals, %d loci, %d reads)" % (len(ivs), loci.n, soa.n))
    prm0 = bench.vc_params(bargs)
    from dataclasses import replace
    prm = replace(prm0, maxMT=1000)
    new = load_lib(None)

    # ---- A. every locus drawn
    # a run that drew keeps its masks: a later run of the same upload applies them and draws nothing, so every run here
    # follows its own upload
    c = new(prm, device_downsample=True)
    for _ in range(2):
        c.upload(soa, loci)
        c.run()
    dev, wall = [], []
    for _ in range(a.runs):
        c.upload(soa, loci)
        t0 = time.perf_counter()
        c.run()
        wall.append(1e3 * (time.perf_counter() - t0))
        dev.append(c.timings()["ms_total_device"])
    res = c.download()
    st = res.loc[_ffi.L_STATUS, :loci.n]
    n_drawn = int(((st & _ffi.ST_DOWNSAMPLED) != 0).sum())
    assert not (st & _ffi.ST_NEED_DOWNSAMPLE).any()
    c_off = new(prm)
    c_off.upload(soa, loci)
    c_off.run()
    dev_flag = []
    for _ in range(a.runs):
        c_off.run()
        dev_flag.append(c_off.timings()["ms_total_device"])
    emit(out, dict(base, leg="A", what="resident run, maxMT=1000, device draw (CUDA events: whole run incl. draw and second pileup)",
                   n_loci_drawn=n_drawn, barcodes_listed=int(res.loc[_ffi.L_NBC, :loci.n][(st & _ffi.ST_DOWNSAMPLED) != 0].sum()),
                   ms_total_device_median=float(np.median(dev)), ms_total_device_min=float(np.min(dev)),
                   ms_wall_run_median=float(np.median(wall)), ms_total_device_flag_only_median=float(np.median(dev_flag)),
                   kernel_launches=int(c.timings()["kernel_launches"])))
    from torch.profiler import ProfilerActivity, profile
    c.upload(soa, loci)
    with profile(activities=[ProfilerActivity.CUDA]) as p:
        c.run()
    kern = sorted((e for e in p.events() if e.device_type == torch.autograd.DeviceType.CUDA and e.device_time > 0), key=lambda e: e.time_range.start)
    names = [e.name for e in kern]
    i0 = next(i for i, nm in enumerate(names) if "k_ds_flags" in nm)
    i1 = max(i for i, nm in enumerate(names) if "k_ds_csr" in nm)
    span_us = kern[i1].time_range.end - kern[i0].time_range.start
    by = {}
    for e in kern[i0:i1 + 1]:
        by[e.name] = by.get(e.name, 0.0) + e.device_time / 1e3
    emit(out, dict(base, leg="A", what="the draw alone (torch.profiler, one run): device span from k_ds_flags to k_ds_csr, kernel ms by name",
                   ms_draw_span=span_us / 1e3, ms_draw_kernels=sum(by.values()),
                   kernels={k[:80]: round(v, 4) for k, v in sorted(by.items(), key=lambda kv: -kv[1])}))
    c.close()

    t0 = time.perf_counter()
    call_loci(full, ivs, refs, prm, gpus=1)
    t_first = time.perf_counter() - t0
    t0 = time.perf_counter()
    rows = call_loci(full, ivs, refs, prm, gpus=1)
    emit(out, dict(base, leg="A", what="call_loci wall time, maxMT=1000, whole reads in, rows out (device draw); second call", rows=len(rows),
                   ms_call_loci=1e3 * (time.perf_counter() - t0), ms_call_loci_first=1e3 * t_first))

    # the parent's host draw on a sample of the flagged loci
    res = c_off.download()
    flagged = np.flatnonzero(res.loc[_ffi.L_STATUS, :loci.n] & _ffi.ST_NEED_DOWNSAMPLE)
    rng = np.random.default_rng(0)
    pick = np.sort(rng.choice(flagged, size=min(a.host_sample, len(flagged)), replace=False))
    st = res.loc[_ffi.L_STATUS]
    st[:loci.n] &= ~_ffi.ST_NEED_DOWNSAMPLE
    st[pick] |= _ffi.ST_NEED_DOWNSAMPLE
    t0 = time.perf_counter()
    keep = draw_keep_masks(c_off, res, soa, loci, soa.chroms, prm)
    t_host = time.perf_counter() - t0
    assert isinstance(keep, UmiKeep) and len(keep.locus) == len(pick)
    per = 1e3 * t_host / len(pick)
    emit(out, dict(base, leg="A", what="host draw (downsample.draw_keep_masks: device listing + Python draw) on a sample of flagged loci; "
                   "the total is an EXTRAPOLATION to all flagged loci, not a measurement",
                   loci_sampled=int(len(pick)), ms_per_locus=per, n_flagged=int(len(flagged)), ms_extrapolated_all_flagged=per * len(flagged)))
    c_off.close()

    # ---- B. nothing flagged: parent / new (mode off) / new (device draw on), alternating
    arms = [("new_flag", new, {}), ("new_device_draw", new, dict(device_downsample=True))]
    if a.parent_lib:
        arms.insert(0, ("parent", load_lib(a.parent_lib), {}))
    callers = {}
    for name, make, kw in arms:
        cc = make(prm0, **kw)
        cc.upload(soa, loci)
        for _ in range(3):
            cc.run()
        callers[name] = cc
    ms = {name: [] for name in callers}
    launches = {}
    for _ in range(a.rounds):
        for name, cc in callers.items():
            for _ in range(a.runs):
                cc.run()
                ms[name].append(cc.timings()["ms_total_device"])
            launches[name] = int(cc.timings()["kernel_launches"])
    outs = {name: cc.download() for name, cc in callers.items()}
    # smc_call_batch (pipelined upload from pageable host buffers, kernels, download), one context per arm, alternating
    call_ms = {name: [] for name in callers}
    for name, cc in callers.items():
        cc.call(soa, loci)
    for _ in range(a.rounds):
        for name, cc in callers.items():
            for _ in range(a.runs // 2):
                t0 = time.perf_counter()
                cc.call(soa, loci)
                call_ms[name].append(1e3 * (time.perf_counter() - t0))

    def same(results):
        # every output array, dynamic-allele rows cut to n_dyn (the representative-read handles name whichever read came first)
        arrs = [{k: v[:r.n_dyn] if k.startswith("dyn_") and k != "dyn_first" else v for k, v in r.__dict__.items()
                 if isinstance(v, np.ndarray) and k not in ("dyn_rep_read", "dyn_rep_qpos")} for r in results.values()]
        return all(x.keys() == arrs[0].keys() and all(np.array_equal(x[k], arrs[0][k], equal_nan=x[k].dtype.kind == "f") for k in x)
                   for x in arrs[1:])
    emit(out, dict(base, leg="B", what="default cfg2 (maxMT=0, nothing flagged): resident ms_total_device, arms alternating %d rounds x %d runs"
                   % (a.rounds, a.runs), **{name + "_median": float(np.median(v)) for name, v in ms.items()},
                   **{name + "_min": float(np.min(v)) for name, v in ms.items()},
                   **{name + "_p90": float(np.percentile(v, 90)) for name, v in ms.items()},
                   **{name + "_call_batch_wall_median": float(np.median(v)) for name, v in call_ms.items()},
                   kernel_launches=launches, outputs_identical=same(outs)))
    for cc in callers.values():
        cc.close()


if __name__ == "__main__":
    main()
