"""Argument checks of smc_upload / smc_call_batch (include/smc_b200.h).  Each malformed batch gets its documented return code
and message from both entry points, and the context that rejected it then computes a valid batch exactly as a fresh
context does."""
from __future__ import annotations

import ctypes as C

import numpy as np
import pytest

from helpers import assert_same_results
from smcounter_b200 import _ffi
from smcounter_b200.caller import GpuCaller, LocusResults, VcParams
from smcounter_b200.synth import SynthSpec, make_panel
from smcounter_b200.targets import build_loci

IVS = [("chr1", 1000, 1100), ("chr1", 1300, 1340)]
PRM = VcParams(mtDepth=20, rpb=3.0)
_STORE = np.zeros(4, np.int32)        # a store_lo / seq_exc array that is given where its partner is not


def _set(**fields):
    def f(rs, ls):
        for k, v in fields.items():
            setattr(rs, k, v)
    return f


def _many_loci(rs, ls):
    ls.n_loci = 4194303


# (name, mutation of the valid (reads, loci) structs, code, message)
CASES = [
    ("negative_n_reads", _set(n_reads=-1), _ffi.SMC_E_ARG, "smc_upload: negative size"),
    ("too_many_loci", _many_loci, _ffi.SMC_E_LIMIT, "smc_upload: more than 4194302 loci in one batch"),
    ("seq_bytes_4gib", _set(seq_bytes=1 << 32), _ffi.SMC_E_LIMIT,
     "smc_upload: batch exceeds 2^30 reads or 4 GiB of bases/qualities/cigar; split the batch"),
    ("scalar_bits", _set(scalar_bits=12), _ffi.SMC_E_ARG, "smc_upload: scalar_bits must be 0, 8, 16 or 32"),
    ("qual_bits", _set(qual_bits=3), _ffi.SMC_E_ARG, "smc_upload: qual_bits must be 0, 2, 4 or 8"),
    ("compact_qual_without_lut", _set(qual_bits=4, qual_lut=None), _ffi.SMC_E_ARG,
     "smc_upload: compact qualities need the packed layout (qual_off == NULL) and a qual_lut"),
    ("seq_bits", _set(seq_bits=3), _ffi.SMC_E_ARG, "smc_upload: seq_bits must be 0, 2 or 4"),
    ("compact_seq_missing_exceptions", _set(seq_bits=2, n_seq_exc=4, seq_exc_read=_STORE.ctypes.data, seq_exc_pos=None,
                                            seq_exc_nib=_STORE.ctypes.data), _ffi.SMC_E_ARG,
     "smc_upload: compact bases need the packed layout (seq_off == NULL) and consistent exception arrays"),
    ("compact_seq_negative_exceptions", _set(seq_bits=2, n_seq_exc=-1), _ffi.SMC_E_ARG,
     "smc_upload: compact bases need the packed layout (seq_off == NULL) and consistent exception arrays"),
    ("ref_id_bits", _set(ref_id_bits=16), _ffi.SMC_E_ARG, "smc_upload: ref_id_bits must be 0, 8 or 32 and umi_bits 0, 32 or 64"),
    ("umi_bits", _set(umi_bits=16), _ffi.SMC_E_ARG, "smc_upload: ref_id_bits must be 0, 8 or 32 and umi_bits 0, 32 or 64"),
    ("store_lo_without_store_len", _set(store_lo=_STORE.ctypes.data, store_len=None), _ffi.SMC_E_ARG,
     "smc_upload: store_lo and store_len must be given together"),
    ("expanded_payload_4gib", _set(seq_bits=2, n_seq_exc=0, seq_bytes=1 << 31), _ffi.SMC_E_LIMIT,
     "smc_upload: the expanded bases / qualities of the batch exceed 4 GiB; split the batch"),
]


@pytest.fixture(scope="module")
def panel():
    soa, refs, _ = make_panel(IVS, SynthSpec(umis_per_locus=40, rpb=3.0, snv_every=25, snv_vaf=0.2, indel_every=40, indel_vaf=0.15), seed=7)
    loci, _ = build_loci(IVS, soa.chroms, refs)
    return soa.repack(), soa.trim_to_targets(IVS).compact(seq_bits_wanted=2), loci


def _rejected(caller, rs, ls, entry):
    if entry == "smc_upload":
        return caller.lib.smc_upload(caller.h, C.byref(rs), C.byref(ls), None)
    o = LocusResults(1, 16).as_struct()          # never written: the batch is rejected before the download
    return caller.lib.smc_call_batch(caller.h, C.byref(rs), C.byref(ls), None, C.byref(o))


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["smc_upload", "smc_call_batch"])
def test_rejected_batches_leave_the_context_usable(panel, entry, monkeypatch):
    packed, compact, loci = panel
    caller = GpuCaller(PRM)
    try:
        for name, mutate, code, msg in CASES:
            for soa in (packed, compact):
                rs, ls = caller._reads_struct(soa), caller._loci_struct(loci)
                mutate(rs, ls)
                rc = _rejected(caller, rs, ls, entry)
                assert (rc, caller.lib.smc_last_error(caller.h).decode()) == (code, msg), (name, soa.seq_bits)
        ls = caller._loci_struct(loci)
        assert caller.lib.smc_upload(caller.h, None, C.byref(ls), None) == _ffi.SMC_E_ARG
        assert caller.lib.smc_last_error(caller.h).decode() == "smc_upload: null reads/loci"
        # the same context after all of the above, against a fresh one: one-chunk and three-chunk uploads, both encodings
        for chunks in ("1", "3"):
            monkeypatch.setenv("SMC_PIPE_CHUNKS", chunks)
            for soa in (packed, compact):
                fresh = GpuCaller(PRM)
                try:
                    want = fresh.call(soa, loci)
                finally:
                    fresh.close()
                if entry == "smc_upload":
                    caller.upload(soa, loci)
                    caller.run()
                    got = caller.download()
                else:
                    got = caller.call(soa, loci)
                    assert caller.timings()["pipe_chunks"] == int(chunks)
                assert_same_results(got, want)
    finally:
        caller.close()
