"""Reads of one fragment that lie far apart in BAM order, through the CUDA path and the oracle.

The device orders the reads by (barcode, frag_id, BAM index) by sorting the fragment ids on their barcode and placing every read
at its fragment's first position plus its rank inside the fragment: a fragment of one or two reads needs only its smallest BAM
index, larger ones take a separate ranking pass.  These batches put R1 and R2 of each fragment far apart, interleaved with the
reads of other fragments and barcodes, add a fragment of exactly three reads, and check that a frag_id shared by two barcodes
is refused."""
from __future__ import annotations

import pytest

from smcounter_b200.caller import VcParams
from test_gpu_hand_built_reads import CONTIGS, Corpus

PRM = VcParams(mtDepth=50, rpb=3.0, minBQ=20, minMQ=30, mismatchThr=6.0, primerDist=2, mtDrop=0)
CHROMS = [name for name, _ in CONTIGS]


def interleaved_mates(three_read_fragment: bool):
    """40 fragments of 8 barcodes on chr1 [1000, 1128): R1 at 1000 + k, R2 at 1040 + (7k mod 40), so that every R2 comes after
    the R1s and R2s of other fragments.  Alternate alleles at 1050 (both mates: concordant) and 1060 (R1 only: discordant)."""
    c = Corpus(seed=23)
    c.group = "mates"
    c.target("chr1", 1000, 1128)
    bcs = [c.barcode() for _ in range(8)]
    for k in range(40):
        bc, rid = bcs[k % 8], "M%d" % k
        both = {1050: "G"} if k % 5 == 0 else {}
        r1_only = {1060: "T"} if k % 3 == 0 else {}
        c.add("r1", "chr1", 1000 + k, "70M", bc, rid, flag=0x40, sub={**both, **r1_only}, qual=30 + k % 8)
        c.add("r2", "chr1", 1040 + (7 * k) % 40, "70M", bc, rid, flag=0x90, sub=both, qual=25 + k % 11)
    if three_read_fragment:
        # R1, R2 and a supplementary R1 alignment far downstream: the BAM order of the three reads is not their arrival order
        bc = bcs[3]
        c.add("triple", "chr1", 1010, "60M", bc, "T0", flag=0x40, sub={1050: "G"}, qual=35)
        c.add("triple", "chr1", 1030, "60M", bc, "T0", flag=0x90, sub={1050: "G"}, qual=33)
        c.add("triple", "chr1", 1085, "40M", bc, "T0", flag=0x840, sub={1100: "C"}, qual=37)
    c.group = None
    return c


def _records_are_interleaved(c):
    """Sanity of the layout: some fragment has reads of other fragments between its two reads in BAM order."""
    names = [r.qname.split(":")[0] for r in c.records()]
    first, last = {}, {}
    for i, q in enumerate(names):
        first.setdefault(q, i)
        last[q] = i
    return max(last[q] - first[q] for q in first) > 20


@pytest.mark.gpu
@pytest.mark.parametrize("three_read_fragment", [False, True])
def test_far_apart_mates_match_oracle(three_read_fragment):
    from helpers import run_records
    c = interleaved_mates(three_read_fragment)
    assert _records_are_interleaved(c)
    problems, stats, (soa, *_rest) = run_records(c.records(), c.intervals["mates"], c.refs(), PRM, chroms=CHROMS)
    print(stats)
    assert stats["events"] > 0
    sizes = sorted(int((soa.frag_id == f).sum()) for f in set(soa.frag_id.tolist()))
    assert sizes[-1] == (3 if three_read_fragment else 2) and sizes[0] == 2
    assert not problems, "\n".join(problems[:30])


@pytest.mark.gpu
def test_fragment_id_with_two_barcodes_is_refused():
    import numpy as np
    from smcounter_b200.caller import GpuCaller
    from smcounter_b200.soa import records_to_soa
    from smcounter_b200.targets import build_loci
    c = interleaved_mates(False)
    ivs = c.intervals["mates"]
    soa = records_to_soa(c.records(), CHROMS)
    loci, _ = build_loci(ivs, soa.chroms, c.refs())
    g = GpuCaller(PRM, 0)
    try:
        g.call(soa, loci)                                    # the unchanged batch is fine
        f0 = np.flatnonzero(soa.frag_id == soa.frag_id[0])
        other = int(np.flatnonzero(soa.umi != soa.umi[0])[0])
        soa.umi = soa.umi.copy()
        soa.umi[f0[-1]] = soa.umi[other]                     # R2 of fragment 0 now carries another fragment's barcode
        with pytest.raises(RuntimeError, match="a frag_id must belong to one barcode"):
            g.call(soa, loci)
    finally:
        g.close()
