"""Shared parity machinery: run the oracle and the CUDA path on the same seeded inputs and diff everything."""
from __future__ import annotations

import math

import numpy as np

from oracle import smcounter_oracle as orc
from smcounter_b200 import _ffi
from smcounter_b200.caller import GpuCaller, LocusResults, UmiKeep, VcParams
from smcounter_b200.rows import AlleleNamer, device_hp_flags, format_rows
from smcounter_b200.soa import soa_to_records
from smcounter_b200.synth import SynthSpec, make_panel
from smcounter_b200.targets import build_loci, loc_list

PI_RTOL = 1e-9       # north_star: PI and p-values within 1e-9 relative
P_RTOL = 1e-9


def oracle_run(soa, intervals, refs, prm: VcParams, keep=None):
    """Rows + per-locus detail dicts from the CPU oracle, in the reference's BED order."""
    recs = soa_to_records(soa, orc.Read)
    index = orc.ReadIndex(recs)
    rows, details = [], []
    for (chrom, pos) in loc_list(intervals):
        d = {}
        k = None if keep is None else keep.get((chrom, pos))
        line = orc.vc(index, chrom, pos, prm.minBQ, prm.minMQ, prm.mtDepth, prm.rpb, prm.hpLen, prm.mismatchThr, prm.mtDrop,
                      prm.maxMT, prm.primerDist, refs, keep_umis=k, detail=d)
        rows.append(line)
        details.append(d)
    return rows, details


def gpu_run(soa, intervals, refs, prm: VcParams, keep: UmiKeep | None = None, device=0):
    loci, bed_order = build_loci(intervals, soa.chroms, refs)
    caller = GpuCaller(prm, device)
    res = caller.call(soa, loci, keep)
    tm = caller.timings()
    hp = device_hp_flags(caller, res, soa, loci, soa.chroms, refs, prm.hpLen)
    caller.close()
    rows = format_rows(res, soa, loci, soa.chroms, refs, prm.hpLen, bed_order, hp_flags=hp)
    return rows, res, loci, bed_order, tm


def rel_err(a, b):
    if a == b:
        return 0.0
    if math.isnan(a) and math.isnan(b):
        return 0.0
    if math.isinf(a) or math.isinf(b) or math.isnan(a) or math.isnan(b):
        return float("inf")
    return abs(a - b) / max(abs(a), abs(b))


def result_arrays(res: LocusResults) -> dict:
    """Every output array of a call, dynamic-allele rows cut to n_dyn, for comparing two calls bit for bit."""
    # the representative-read handles of dynamic alleles name whichever read reached the device table first
    skip = ("dyn_rep_read", "dyn_rep_qpos")
    out = {k: v[: res.n_dyn] if k.startswith("dyn_") and k != "dyn_first" else v
           for k, v in res.__dict__.items() if isinstance(v, np.ndarray) and k not in skip}
    out["n_dyn"] = np.array([res.n_dyn])
    return out


def assert_same_results(a: LocusResults, b: LocusResults):
    ra, rb = result_arrays(a), result_arrays(b)
    assert ra.keys() == rb.keys()
    for k in ra:
        assert np.array_equal(ra[k], rb[k], equal_nan=ra[k].dtype.kind == "f"), k


def diff_details(res, loci, bed_order, details, soa, refs, max_report=20):
    """Field-by-field diff of the device results against the oracle's detail dicts.  Returns (problems, stats)."""
    namer = AlleleNamer(res, soa, loci, soa.chroms, refs)
    problems = []
    max_pi_err = 0.0
    max_p_err = 0.0
    n_fisher = 0
    counter_map = (("alleleCnt", _ffi.C_ALLELE), ("forwardCnt", _ffi.C_FWD), ("reverseCnt", _ffi.C_REV), ("lowQReads", _ffi.C_LOWQ),
                   ("r1Le", _ffi.C_R1LE), ("r1Tot", _ffi.C_R1TOT), ("r2Le", _ffi.C_R2LE), ("r2Tot", _ffi.C_R2TOT),
                   ("r2PLe", _ffi.C_R2PLE), ("concord", _ffi.C_CONCORD), ("discord", _ffi.C_DISCORD), ("MTCnt", _ffi.C_MT),
                   ("strongMTCnt", _ffi.C_STRONG))
    for k, d in enumerate(details):
        i = int(bed_order[k])

        def bad(msg):
            if len(problems) < max_report:
                problems.append("locus %d (%s:%d): %s" % (i, soa.chroms[int(loci.ref_id[i])], int(loci.pos0[i]) + 1, msg))

        for name, idx in (("cvg", _ffi.L_CVG), ("allFrag", _ffi.L_ALLFRAG), ("allMT", _ffi.L_ALLMT), ("nBC", _ffi.L_NBC)):
            if int(res.loc[idx, i]) != d[name]:
                bad("%s gpu=%d oracle=%d" % (name, int(res.loc[idx, i]), d[name]))
        if "usedMT" not in d:      # zero coverage
            if not (int(res.loc[_ffi.L_STATUS, i]) & _ffi.ST_ZERO_COVERAGE):
                bad("oracle says zero coverage, gpu status=%d" % int(res.loc[_ffi.L_STATUS, i]))
            continue
        for name, idx in (("usedMT", _ffi.L_USEDMT), ("usedFrag", _ffi.L_USEDFRAG), ("MT3", _ffi.L_MT3), ("MT5", _ffi.L_MT5),
                          ("MT7", _ffi.L_MT7), ("MT10", _ffi.L_MT10)):
            if int(res.loc[idx, i]) != d[name]:
                bad("%s gpu=%d oracle=%d" % (name, int(res.loc[idx, i]), d[name]))
        # allele name -> reference
        refs_by_name = {n: a for a, n in enumerate(_ffi.FIXED_NAMES)}
        d0, d1 = int(res.dyn_first[i]), int(res.dyn_first[i + 1])
        for j in range(d0, d1):
            refs_by_name[namer.name(_ffi.SMC_NFIXED + j)] = _ffi.SMC_NFIXED + j

        def cnt(a, c):
            return int(res.cnt[a, c, i]) if a < _ffi.SMC_NFIXED else int(res.dyn_cnt[a - _ffi.SMC_NFIXED, c])

        for al in d["alleles"]:
            if al not in refs_by_name:
                bad("allele %s missing on gpu" % al)
                continue
            a = refs_by_name[al]
            for name, c in counter_map:
                want = d[name].get(al, 0)
                if cnt(a, c) != want:
                    bad("%s[%s] gpu=%d oracle=%d" % (name, al, cnt(a, c), want))
            if al in d["PI"]:
                got = float(res.pi[a, i]) if a < _ffi.SMC_NFIXED else float(res.dyn_pi[a - _ffi.SMC_NFIXED])
                e = rel_err(got, d["PI"][al])
                max_pi_err = max(max_pi_err, e)
                if e > PI_RTOL:
                    bad("PI[%s] gpu=%r oracle=%r" % (al, got, d["PI"][al]))
        for al, a in refs_by_name.items():
            if al not in d["alleles"] and any(cnt(a, c) for _, c in counter_map):
                bad("gpu has counts for allele %s unknown to the oracle" % al)
        for name, arr in (("maxBase", res.max_allele), ("secondMaxBase", res.second_allele), ("firstAlt", res.alt_allele)):
            got = namer.name(int(arr[i]))
            if got != d[name]:
                bad("%s gpu=%s oracle=%s" % (name, got, d[name]))
        e = rel_err(float(res.alt_pi[i]), d["altPI"])
        if e > PI_RTOL:
            bad("altPI gpu=%r oracle=%r" % (float(res.alt_pi[i]), d["altPI"]))
        if bool(res.biallelic[i]) != d["biallelic"]:
            bad("biallelic gpu=%d oracle=%d" % (int(res.biallelic[i]), d["biallelic"]))
        for cand, fd in ((0, d["filt1"]), (1, d["filt2"])):
            for t, key in ((0, "sb"), (1, "r1"), (2, "r2"), (3, "primer")):
                gp, go = float(res.fisher_p[cand, t, i]), float(res.fisher_or[cand, t, i])
                if key in fd:
                    n_fisher += 1
                    _, oo, op = fd[key]
                    ep = rel_err(gp, op)
                    max_p_err = max(max_p_err, ep)
                    if ep > P_RTOL:
                        bad("fisher p %s cand%d table=%s gpu=%r oracle=%r" % (key, cand, fd[key][0], gp, op))
                    if rel_err(go, oo) > 1e-12:
                        bad("fisher OR %s cand%d table=%s gpu=%r oracle=%r" % (key, cand, fd[key][0], go, oo))
                elif not math.isnan(gp):
                    bad("gpu evaluated fisher %s cand%d but the oracle did not" % (key, cand))
    return problems, dict(max_pi_rel_err=max_pi_err, max_p_rel_err=max_p_err, n_fisher=n_fisher)


def diff_rows(gpu_rows, oracle_rows, max_report=10):
    out = []
    for k, (g, o) in enumerate(zip(gpu_rows, oracle_rows)):
        if g != o:
            gf, of = g.split("\t"), o.split("\t")
            cols = [(orc.headerAll[c], gf[c], of[c]) for c in range(min(len(gf), len(of))) if gf[c] != of[c]]
            out.append("row %d %s:%s differs: %s" % (k, of[0], of[1], cols[:8]))
            if len(out) >= max_report:
                break
    if len(gpu_rows) != len(oracle_rows):
        out.append("row count gpu=%d oracle=%d" % (len(gpu_rows), len(oracle_rows)))
    return out


def keep_from_oracle(details, bed_order, soa):
    """The read-selection mask the oracle produced (north_star: 'subsampling taken from the same mask'): for every
    locus where down-sampling fired, the barcodes the oracle kept, as 64-bit codes."""
    from smcounter_b200.soa import umi_code
    table = {}
    if soa.umi_names:
        inv = {v: k for k, v in soa.umi_names.items()}
    else:
        inv = None
    mapping = {}
    for k, d in enumerate(details):
        if "usedMT" in d and d["nBC"] > d["ds"]:
            codes = [(inv[bc] if inv is not None else umi_code(bc, table)) for bc in d["bcKeys"]]
            mapping[int(bed_order[k])] = codes
    return UmiKeep(mapping) if mapping else None


def run_case(intervals, spec: SynthSpec, prm: VcParams, seed: int, verbose=False, mutate=None, gpu_mutate=None):
    """``mutate``: applied to the generated reads before both sides see them; ``gpu_mutate``: a different ENCODING of the same
    reads for the CUDA path only (packed, trimmed to the targets, ...) -- the oracle keeps the plain one."""
    soa, refs, truth = make_panel(intervals, spec, seed=seed)
    if mutate is not None:
        soa = mutate(soa)
    o_rows, details = oracle_run(soa, intervals, refs, prm)
    _, bo = build_loci(intervals, soa.chroms, refs)
    keep = keep_from_oracle(details, bo, soa)
    gsoa = gpu_mutate(soa) if gpu_mutate is not None else soa
    g_rows, res, loci, bed_order, tm = gpu_run(gsoa, intervals, refs, prm, keep)
    problems, stats = diff_details(res, loci, bed_order, details, gsoa, refs)
    problems += diff_rows(g_rows, o_rows)
    stats.update(n_downsampled=0 if keep is None else len(keep.locus), n_reads=soa.n, payload_bytes=int(gsoa.seq.nbytes + gsoa.qual.nbytes), n_loci=loci.n, events=tm["n_pileup_events"], n_dyn=tm["n_dyn"], code_mult=tm["code_mult"], dyn_capacity=tm["dyn_capacity"], pipe_chunks=tm["pipe_chunks"], pipe_launches=tm["pipe_launches"], ms_device=tm["ms_total_device"],
                 ms_pileup=tm["ms_pileup"])
    if verbose:
        print(stats)
        for p in problems:
            print("  ", p)
    return problems, stats, (soa, refs, o_rows, g_rows, res, details)


def run_records(records, intervals, refs, prm: VcParams, chroms=None, verbose=False):
    """Hand-made reads (oracle.Read records in BAM order) through the CUDA path and the oracle: (problems, stats, extras)."""
    from smcounter_b200.soa import records_to_soa
    soa = records_to_soa(records, chroms)
    index = orc.ReadIndex(records)
    o_rows, details = [], []
    for (chrom, pos) in loc_list(intervals):
        d = {}
        o_rows.append(orc.vc(index, chrom, pos, prm.minBQ, prm.minMQ, prm.mtDepth, prm.rpb, prm.hpLen, prm.mismatchThr, prm.mtDrop,
                             prm.maxMT, prm.primerDist, refs, detail=d))
        details.append(d)
    g_rows, res, loci, bed_order, tm = gpu_run(soa, intervals, refs, prm)
    problems, stats = diff_details(res, loci, bed_order, details, soa, refs)
    problems += diff_rows(g_rows, o_rows)
    stats.update(n_dyn=tm["n_dyn"], events=tm["n_pileup_events"])
    if verbose:
        print(stats)
        for p in problems:
            print("  ", p)
    return problems, stats, (soa, o_rows, g_rows, res, details)
