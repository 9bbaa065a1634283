"""Stages of a batch run (smc_run_resident, reached through smc_call_batch) that other tests do not reach: the regrowth of the
tile-event buffers and of the Fisher task list, the device-side input checks on l_seq and on the packed payload size, and the
barcode count smc_timings reports.  Every case runs on a fresh context, with a one-chunk and with a three-chunk upload."""
from __future__ import annotations

import ctypes as C
import dataclasses

import numpy as np
import pytest

from helpers import assert_same_results, keep_from_oracle, run_case
from smcounter_b200 import _ffi
from smcounter_b200.caller import GpuCaller, LocusResults, VcParams
from smcounter_b200.synth import SynthSpec, make_panel
from smcounter_b200.targets import build_loci

pytestmark = [pytest.mark.gpu, pytest.mark.parametrize("chunks", ["1", "3"])]


def _oracle_then_twice(ivs, spec, prm, seed):
    """The batch against the oracle (run_case), then twice on one fresh context: both calls must equal the run_case results.
    Returns the reads and the timings of the fresh context's first call."""
    problems, _, (soa, refs, _o_rows, _g_rows, want, details) = run_case(ivs, spec, prm, seed)
    assert not problems, "\n".join(problems)
    loci, bed_order = build_loci(ivs, soa.chroms, refs)
    keep = keep_from_oracle(details, bed_order, soa)
    caller = GpuCaller(prm)
    try:
        first = caller.call(soa, loci, keep)
        tm = caller.timings()
        assert_same_results(first, want)
        assert_same_results(caller.call(soa, loci, keep), want)    # the buffers have grown: no second regrowth
    finally:
        caller.close()
    return soa, tm


def test_tile_event_buffers_grow(chunks, monkeypatch):
    """300-base reads over a 600-base target cover about seven 32-locus tiles each: more tile events than the first guess of
    4 per read + 4096, so k_expand_scan runs a second time into grown buffers."""
    monkeypatch.setenv("SMC_PIPE_CHUNKS", chunks)
    spec = SynthSpec(read_len=300, umis_per_locus=200, rpb=3.0, snv_every=50, snv_vaf=0.1)
    soa, tm = _oracle_then_twice([("chr1", 1000, 1600)], spec, VcParams(mtDepth=200, rpb=3.0), seed=89)
    assert tm["pipe_chunks"] == int(chunks)
    assert tm["n_tile_events"] > 4 * soa.n + 4096, "the input no longer outgrows the first tile-event buffers"


def test_fisher_task_list_grows(chunks, monkeypatch):
    """An SNV at every target base (mismatch filter off): more Fisher tests than the first task list of 8192 holds, so k_call,
    k_fisher and k_sum_cvg run a second time."""
    monkeypatch.setenv("SMC_PIPE_CHUNKS", chunks)
    ivs = [("chr1", 1000, 2000), ("chr2", 1000, 2000), ("chr3", 1000, 2000)]
    spec = SynthSpec(umis_per_locus=20, rpb=2.0, snv_every=1, snv_vaf=0.3)
    _, tm = _oracle_then_twice(ivs, spec, VcParams(mtDepth=20, rpb=2.0, mismatchThr=100.0), seed=83)
    assert tm["pipe_chunks"] == int(chunks)
    assert tm["n_fisher"] > 8192, "the input no longer outgrows the first Fisher task list"


IVS = [("chr1", 1000, 1100), ("chr1", 1300, 1340)]
PRM = VcParams(mtDepth=20, rpb=3.0)


@pytest.fixture(scope="module")
def panel():
    soa, refs, _ = make_panel(IVS, SynthSpec(umis_per_locus=40, rpb=3.0, snv_every=25, snv_vaf=0.2, indel_every=40, indel_vaf=0.15), seed=7)
    loci, _ = build_loci(IVS, soa.chroms, refs)
    return soa, loci


def _long_read(soa):
    """One read claims 70000 bases; its offsets stay valid, so nothing is read past the caller's arrays."""
    l_seq = soa.l_seq.copy()
    l_seq[soa.n // 2] = 70000
    return soa, dataclasses.replace(soa, l_seq=l_seq)


def _short_packed_payload(soa):
    """Packed bases (NULL offsets) declared two bytes shorter than the per-read lengths add up to."""
    good = soa.repack()
    return good, dataclasses.replace(good, seq=good.seq[:-2])


@pytest.mark.parametrize("make, code, msg", [
    (_long_read, _ffi.SMC_E_LIMIT, "a read has l_seq or clip length > 65535 (unsupported)"),
    (_short_packed_payload, _ffi.SMC_E_ARG, "packed payload (NULL offsets): seq_bytes / qual_bytes / n_cigar_words do not match the sums "
                                            "of (len+1)/2, len, n_cigar (len = store_len or l_seq)"),
], ids=["l_seq_over_65535", "packed_seq_bytes_short"])
def test_device_side_checks_leave_the_context_usable(panel, make, code, msg, chunks, monkeypatch):
    monkeypatch.setenv("SMC_PIPE_CHUNKS", chunks)
    soa, loci = panel
    good, bad = make(soa)
    fresh = GpuCaller(PRM)
    try:
        want = fresh.call(good, loci)
    finally:
        fresh.close()
    caller = GpuCaller(PRM)
    try:
        rs, ls = caller._reads_struct(bad), caller._loci_struct(loci)
        o = LocusResults(loci.n, 16).as_struct()          # never written: the batch is rejected before the download
        rc = caller.lib.smc_call_batch(caller.h, C.byref(rs), C.byref(ls), None, C.byref(o))
        assert (rc, caller.lib.smc_last_error(caller.h).decode()) == (code, msg)
        got = caller.call(good, loci)
        assert caller.timings()["pipe_chunks"] == int(chunks)
        assert_same_results(got, want)
    finally:
        caller.close()


def test_n_umi_groups_counts_the_barcodes(panel, chunks, monkeypatch):
    """n_umi_groups is the number of distinct barcodes of the batch; 0 when the read sort does not run (no reads or no loci),
    also on a context whose previous batch had barcodes."""
    monkeypatch.setenv("SMC_PIPE_CHUNKS", chunks)
    soa, loci = panel
    no_loci, _ = build_loci([], soa.chroms, {})
    caller = GpuCaller(PRM)
    try:
        caller.call(soa, loci)
        assert caller.timings()["n_umi_groups"] == np.unique(soa.umi).size > 0
        caller.call(soa.select(np.zeros(0, dtype=np.int64)), loci)
        assert caller.timings()["n_umi_groups"] == 0
        caller.call(soa, no_loci)
        assert caller.timings()["n_umi_groups"] == 0
    finally:
        caller.close()
