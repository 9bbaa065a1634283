"""The device keeps one 16-bit word (quality | base nibble << 8) per stored base, sized from the declared payload bytes.  A caller
that gives its own offsets can declare fewer bytes than its reads' lengths need (reads sharing payload bytes); such a batch is
refused by the run instead of being expanded past the words the upload provided."""
from __future__ import annotations

import numpy as np
import pytest

from smcounter_b200.caller import GpuCaller, VcParams
from smcounter_b200.synth import SynthSpec, make_panel
from smcounter_b200.targets import build_loci

IVS = [("chr1", 1000, 1100)]


@pytest.mark.gpu
def test_explicit_offsets_sharing_payload_bytes_are_refused():
    soa, refs, _ = make_panel(IVS, SynthSpec(umis_per_locus=20, rpb=3.0), seed=11)
    loci, _ = build_loci(IVS, soa.chroms, refs)
    lmax = int(soa.l_seq.max())
    soa.seq_off = np.zeros(soa.n, np.int64)          # every read points at the first read's bytes
    soa.qual_off = np.zeros(soa.n, np.int64)
    soa.seq = np.ascontiguousarray(soa.seq[:(lmax + 1) // 2])
    soa.qual = np.ascontiguousarray(soa.qual[:lmax])
    soa.packed = False
    caller = GpuCaller(VcParams(mtDepth=20, rpb=3.0))
    try:
        caller.upload(soa, loci)
        with pytest.raises(RuntimeError, match="need more room than seq_bytes provides"):
            caller.run()
    finally:
        caller.close()
