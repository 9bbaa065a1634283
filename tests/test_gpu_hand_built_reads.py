"""Hand-built reads through the CUDA path and the oracle: the CIGAR ops, flags, fragment shapes and long insertions that the
synthetic panels (smcounter_b200/synth.py: M, S M, M S, M I M, M D M, one R1 and one R2 per fragment) never produce, but a
real BAM does.

The corpus is laid out by ``build_corpus()`` on its own reference (``orc.DictFasta``): every case is a few reads at loci the
builder chose, in BAM order, named ``<readid>:<barcode>:<x>``.  Each group of cases is called through every upload encoding
(plain, repack(), trim_to_targets(), trim_to_targets().compact() with 2- and 4-bit bases), one- and three-chunk uploads and two
parameter sets, and diffed against the oracle: every tally bit-exact, PI and Fisher p within 1e-9, rows byte-identical.

Without -m gpu: the oracle's pileup_column() against hand-derived (qpos, indel, is_del) for every new CIGAR shape, a Python
port of the device's long-insertion hash that pins the colliding insertions the corpus relies on, and checks that the corpus
means what it says (BAM order, dense fragment ids, the intended alleles and counts in the oracle's own tallies)."""
from __future__ import annotations

import functools
import os
import random
from collections import defaultdict

import pytest

from oracle import smcounter_oracle as orc
from smcounter_b200.caller import VcParams
from smcounter_b200.targets import loc_list

OPS = "MIDNSHP=X"
CONTIGS = (("chr1", 6000), ("chr2", 1200))
NT16 = "=ACMGRSVTWYHKDBN"

# Insertions longer than 8 bases are keyed by a 32-bit FNV-1a hash (smc_pileup.cuh, slow_event): pairs that collide.
# The first two differ by one trailing base (the length is in the hash seed but not in the key); the third has equal lengths.
COLLIDING_INSERTIONS = (
    ("ATAGCGCCTTGTATAA", "ATAGCGCCTTGTATAAA", 0x6d52e690),
    ("CAATAAAGTTCACAATT", "CAATAAAGTTCACAATTA", 0xe1d24d3a),
    ("AACCACGGTT", "TAGAGCATGC", 0x1e882536),
)

PARAMS = {
    "p1": VcParams(mtDepth=50, rpb=3.0, minBQ=20, minMQ=30, mismatchThr=6.0, primerDist=2, mtDrop=0),
    "p2": VcParams(mtDepth=50, rpb=3.0, minBQ=20, minMQ=30, mismatchThr=6.0, primerDist=2, mtDrop=1, hpLen=8),
}


def long_ins_hash(ins: str) -> int:
    """The device's key of an insertion longer than 8 bases: FNV-1a over BAM nibbles (A1 C2 G4 T8 N15), seeded with the length."""
    h = 2166136261 ^ len(ins)
    for ch in ins:
        h = ((h ^ NT16.index(ch)) * 16777619) & 0xFFFFFFFF
    return h


def parse_cigar(s):
    out, num = [], ""
    for ch in s:
        if ch.isdigit():
            num += ch
        else:
            out.append((OPS.index(ch), int(num)))
            num = ""
    return out


class Corpus:
    """Reads laid out on a seeded random reference.  ``add()`` derives the read's bases from the reference along its CIGAR
    (M / = copy, X substitutes, I takes the given bases, S random ones), with per-position overrides ``sub``; NM defaults to
    mismatches + inserted + deleted bases."""

    def __init__(self, seed=11):
        self.rng = random.Random(seed)
        self.ref = {c: [self.rng.choice("ACGT") for _ in range(n)] for c, n in CONTIGS}
        self.entries = []                 # (contig index, pos, serial, group, case, Read)
        self.intervals = defaultdict(list)
        self.n_bc = 0
        self.group = None

    def set_ref(self, chrom, pos, bases):
        for k, b in enumerate(bases):
            self.ref[chrom][pos + k] = b

    def refs(self):
        return orc.DictFasta({c: "".join(v) for c, v in self.ref.items()})

    def barcode(self):
        self.n_bc += 1
        n = self.n_bc
        return "GT" + "".join("ACGT"[(n >> (2 * k)) & 3] for k in range(10))

    def target(self, chrom, s, e):
        assert (e - s) % 32 == 0          # every interval starts a 32-locus tile (the loci are sorted, intervals disjoint)
        self.intervals[self.group].append((chrom, s, e))

    def rand_bases(self, n):
        return "".join(self.rng.choice("ACGT") for _ in range(n))

    def add(self, case, chrom, pos, cigar, bc, rid, flag=0x40, mapq=60, nm=None, ins=(), sub=None, qual=30, bq=None, seq=None):
        cig = parse_cigar(cigar) if isinstance(cigar, str) else list(cigar)
        ref = self.ref[chrom]
        sub, bq, ins = sub or {}, bq or {}, list(ins)
        s, qref = [], []
        x, mism, nind = pos, 0, 0
        for op, l in cig:
            if op in (0, 7):
                for k in range(l):
                    b = sub.get(x + k, ref[x + k])
                    s.append(b); qref.append(x + k)
                    mism += b != ref[x + k]
                x += l
            elif op == 8:
                for k in range(l):
                    s.append("ACGT"[("ACGT".index(ref[x + k]) + 1) % 4]); qref.append(x + k)
                mism += l
                x += l
            elif op == 1:
                b = ins.pop(0) if ins else self.rand_bases(l)
                assert len(b) == l
                s.extend(b); qref.extend([None] * l)
                nind += l
            elif op == 4:
                s.extend(self.rand_bases(l)); qref.extend([None] * l)
            elif op in (2, 3):
                nind += l if op == 2 else 0
                x += l
        if seq is not None:
            s, qref = list(seq), [None] * len(seq)
        quals = list(qual) if isinstance(qual, (list, tuple)) else [qual] * len(s)
        for i, p in enumerate(qref):
            if p is not None and p in bq:
                quals[i] = bq[p]
        assert len(quals) == len(s)
        r = orc.Read("%s:%s:%d" % (rid, bc, 2 if flag & 0x80 else 1), chrom, pos, flag, mapq, mism + nind if nm is None else nm, cig,
                     "".join(s), quals)
        cidx = [c for c, _ in CONTIGS].index(chrom)
        self.entries.append((cidx, pos, len(self.entries), self.group, case, r))
        return r

    def pair(self, case, chrom, pos, cigar, bc=None, rev1=False, ins=None, **kw):
        """R1 and R2 with the same alignment on opposite strands: one fragment of a new (or the given) barcode."""
        bc = bc or self.barcode()
        if ins is None:
            ins = [self.rand_bases(l) for op, l in parse_cigar(cigar) if op == 1]
        rid = "P%d" % len(self.entries)
        self.add(case, chrom, pos, cigar, bc, rid, flag=0x40 | (0x10 if rev1 else 0), ins=ins, **kw)
        self.add(case, chrom, pos, cigar, bc, rid, flag=0x80 | (0 if rev1 else 0x10), ins=ins, **kw)
        return bc

    def both_strands(self, case, chrom, pos, cigar, **kw):
        """Two fragments of one new barcode: the shape as R1 forward / R2 reverse and as R1 reverse / R2 forward (every
        end-distance formula of smCounter.py:578-594)."""
        ins = kw.pop("ins", None) or [self.rand_bases(l) for op, l in parse_cigar(cigar) if op == 1]
        bc = self.pair(case, chrom, pos, cigar, rev1=False, ins=ins, **kw)
        self.pair(case, chrom, pos, cigar, bc=bc, rev1=True, ins=ins, **kw)

    def records(self, group=None):
        """oracle.Read records in BAM order: sorted by (contig, pos), stable."""
        return [e[5] for e in sorted(self.entries, key=lambda e: (e[0], e[1], e[2])) if group is None or e[3] == group]

    def cases(self, group=None):
        return {e[4] for e in self.entries if group is None or e[3] == group}

    def all_intervals(self):
        return [iv for g in GROUPS for iv in self.intervals[g]]


def _cigar_zoo(c):
    c.group = "cigar"
    c.target("chr1", 1000, 1128)                  # tiles start at 1000, 1032, 1064, 1096
    c.both_strands("H_S_M", "chr1", 1005, "5H10S40M")
    c.both_strands("M_S_H", "chr1", 1010, "40M10S5H")
    c.both_strands("H_M_H", "chr1", 1025, "3H45M4H")
    c.both_strands("eq_X", "chr1", 1020, "30=1X40=")
    c.both_strands("M_eq_X_M", "chr1", 1040, "10M20=1X30=10M")
    c.both_strands("multi_indel", "chr1", 1040, "20M2I15M3D20M1I10M")
    c.both_strands("S_I_M", "chr1", 1050, "5S3I40M")
    c.both_strands("M_I_S", "chr1", 1060, "40M2I6S")
    c.both_strands("M_D_last", "chr1", 1070, "35M4D")
    c.both_strands("D_I", "chr1", 1002, "20M2D3I20M")
    c.both_strands("I_D", "chr1", 1008, "20M3I2D20M")
    c.both_strands("N_skip", "chr1", 1030, "15M40N15M")               # 40 loci inside the skip, across the 1064 boundary
    c.both_strands("N_skip_short", "chr1", 1085, "6M3N20M")
    c.both_strands("M_P_I_M", "chr1", 1015, "25M2P3I25M")
    c.both_strands("M_I_P_I_M", "chr1", 1033, "25M2I1P3I25M")
    c.both_strands("D_across_tile", "chr1", 1010, "20M6D20M")          # deletes 1030..1035
    c.add("no_cigar", "chr1", 1050, [], c.barcode(), "NC1", flag=0x40, seq="ACGTTGCAACGTTGCAACGTTGCAAC", nm=0)
    c.add("no_cigar", "chr1", 1052, [], c.barcode(), "NC2", flag=0x90, seq="ACGTTGCAAC", nm=0)
    for k in range(4):                                                  # plain background with a few SNVs
        c.pair("background", "chr1", 1000 + 19 * k, "60M", rev1=bool(k & 1), sub={1100: "T", 1040: "C"} if k == 2 else None)


def _flag_zoo(c):
    c.group = "flags"
    c.target("chr1", 2000, 2064)
    ref = c.ref["chr1"]
    alt = lambda p: "ACGT"[("ACGT".index(ref[p]) + 2) % 4]
    for k in range(3):
        c.pair("background", "chr1", 2000 + 7 * k, "50M", rev1=bool(k & 1))
    bc = c.barcode()
    c.add("secondary", "chr1", 2005, "40M", bc, "S1", flag=0x140, sub={2030: alt(2030)})
    c.add("secondary", "chr1", 2005, "40M", bc, "S1", flag=0x90, sub={2030: alt(2030)})
    c.add("qcfail", "chr1", 2010, "40M", c.barcode(), "Q1", flag=0x240 | 0x10, sub={2030: alt(2030)})
    c.add("duplicate", "chr1", 2015, "40M", c.barcode(), "D1", flag=0x480, sub={2031: alt(2031)})
    bc = c.barcode()
    c.add("supplementary", "chr1", 2020, "20H40M", bc, "X1", flag=0x840, sub={2031: alt(2031)})
    c.add("supplementary", "chr1", 2022, "40M", bc, "X1", flag=0x90)
    c.add("unmapped", "chr1", 2025, "40M", c.barcode(), "U1", flag=0x44, sub={2033: alt(2033)})        # a barcode seen only here
    c.add("unmapped", "chr1", 2026, "40M", bc, "U2", flag=0x84)                                      # a new fragment of a barcode
    bc_u = c.barcode()
    c.add("unmapped", "chr1", 2012, "40M", bc_u, "U3", flag=0x48)                                   # mate unmapped, placed first
    c.add("unmapped", "chr1", 2013, "40M", bc_u, "U3", flag=0x98)
    c.add("both_r1_r2", "chr1", 2030, "30M", c.barcode(), "B1", flag=0xC0)
    c.add("both_r1_r2", "chr1", 2031, "30M", c.barcode(), "B2", flag=0xD0)
    c.add("both_r1_r2", "chr1", 2004, "20M1D20M", c.barcode(), "B3", flag=0xC0)
    c.add("both_r1_r2", "chr1", 2006, "3S20M2I20M", c.barcode(), "B4", flag=0xD0)
    c.pair("mapq255", "chr1", 2008, "45M", mapq=255)
    c.pair("nm_below_indel", "chr1", 2012, "20M5D20M", nm=2)
    c.pair("nm_below_indel", "chr1", 2014, "20M4I20M", nm=1)
    c.pair("mapq_at_minMQ", "chr1", 2018, "40M", mapq=30, sub={2040: alt(2040)})
    c.pair("mapq_at_minMQ", "chr1", 2019, "40M", mapq=29, sub={2040: alt(2040)})
    # base quality exactly minBQ at even positions, one below at odd ones; an insertion anchored on either
    c.add("bq_at_minBQ", "chr1", 2002, "40M", c.barcode(), "Q20", flag=0x40, bq={p: 20 if p % 2 == 0 else 19 for p in range(2002, 2042)},
          sub={2036: alt(2036), 2037: alt(2037)})
    c.add("bq_at_minBQ", "chr1", 2016, "20M2I20M", c.barcode(), "Q21", flag=0x90, qual=20)
    c.add("bq_at_minBQ", "chr1", 2016, "20M2I20M", c.barcode(), "Q22", flag=0x40, qual=19)
    # 9 mismatches in 150 bases: mm100 == 6.0 == mismatchThr (included); 10: excluded
    c.pair("mm_at_threshold", "chr1", 1950, "150M", nm=9, sub={2045: alt(2045)})
    c.pair("mm_at_threshold", "chr1", 1955, "150M", nm=10, rev1=True, sub={2045: alt(2045)})
    # reads that are not one plain run, fully inside the targets: every end distance 0..alnlen, 20 and primerDist included
    for cig, p in (("2S25M2D25M", 2003), ("5H30M1I20M3S", 2009)):
        c.both_strands("end_dist_not_plain", "chr1", p, cig)


def _read_lengths(c):
    c.group = "lengths"
    c.target("chr1", 3000, 3064)
    c.target("chr1", 3960, 3992)
    c.add("len1", "chr1", 3010, "1M", c.barcode(), "L1", flag=0x40)
    c.add("len2", "chr1", 3031, "2M", c.barcode(), "L2", flag=0x90)                    # across the tile boundary at 3032
    c.pair("len33", "chr1", 3016, "33M", sub={3040: "N"})
    c.pair("len151", "chr1", 2950, "151M", rev1=True)
    c.add("len300", "chr1", 2900, "300M", c.barcode(), "L300", flag=0x50, qual=[12 + (k * 7) % 30 for k in range(300)])
    c.add("len300", "chr1", 2940, "5S140M1I150M4S", c.barcode(), "L300b", flag=0x80)
    c.add("len1000", "chr1", 2990, "1000M", c.barcode(), "L1000", flag=0x80, sub={3000: "N", 3985: "G" if c.ref["chr1"][3985] != "G" else "C"})
    c.add("len1000", "chr1", 2975, "10S990M", c.barcode(), "L1000b", flag=0x50)
    for k in range(3):
        c.pair("background", "chr1", 2995 + 11 * k, "60M", rev1=bool(k & 1))


FZ_LOCUS = 511                         # chr2: last locus of the first tile of [480, 544); 512 starts the next


def _fragment_zoo(c):
    c.group = "fragments"
    c.target("chr2", 480, 544)
    c.set_ref("chr2", FZ_LOCUS, "A")
    rng = random.Random(5)
    # one barcode, 64 fragments of 1, 2, 3, 4 reads (cycling): fragment starts fall on every offset of a 32-event batch
    z1 = c.barcode()
    patterns = {1: (("A",), ("G",)),
                2: (("A", "A"), ("A", "G")),
                3: (("A", "A", "A"), ("A", "G", "G"), ("A", "N", "A")),          # concordant; discordant then recreated; N kept
                4: (("N", "A", "A", "A"), ("R", "R", "Y", "R"), ("G", "G", "G", "G"))}
    flags = (0x40, 0x90, 0x840, 0x190)                                           # R1, R2, supplementary R1, secondary R2
    for f in range(64):
        size = f % 4 + 1
        bases = patterns[size][(f // 4) % len(patterns[size])]
        pos = 480 + (f * 5) % 24
        rid = "Z1F%d" % f
        for k, b in enumerate(bases):
            q = (15, 25, 33, 38)[(f + k) % 4]
            c.add("frag_size_%d" % size, "chr2", pos, "40M", z1, rid, flag=flags[k], sub={FZ_LOCUS: b},
                  qual=[rng.choice((20, 30, 37)) for _ in range(40)], bq={FZ_LOCUS: q})
    # one fragment of 45 reads at one locus: carried across batches; a G deletes it in the middle, the next A recreates it
    z2 = c.barcode()
    for k in range(45):
        b = "G" if k == 17 else "N" if k == 30 else "A"
        c.add("frag_45_reads", "chr2", 495, "35M", z2, "Z2F0", flag=(0x40, 0x90, 0x140, 0x190)[min(k, 2 + (k & 1))],
              sub={FZ_LOCUS: b}, qual=20 + k % 20)
    # a barcode with a non-ACGT character: dictionary-coded (stays 64-bit in compact())
    zn = "ACNTGACTGACT"
    for f in range(3):
        c.pair("barcode_with_N", "chr2", 488 + f, "40M", bc=zn, sub={FZ_LOCUS: "G"} if f == 1 else None)
    for k in range(6):
        c.pair("background", "chr2", 482 + 3 * k, "45M", rev1=bool(k & 1), sub={FZ_LOCUS: "G"} if k < 2 else None)


LONG_INS = {"ins9": "GATTACAGG", "ins16": "TTGACCAGTACGGATC", "ins31N": "ACCGTTAGCATGNCAGTTACGGATCATGCAA", "ins12": "CTTAGGACCATG"}


def _long_insertions(c):
    c.group = "long_ins"
    c.target("chr1", 5000, 5064)
    # (anchor, [(insertion, supporting barcodes)]): distinct counts for distinct alleles, no exact PI ties
    sites = [(5010, [(LONG_INS["ins9"], 4), (LONG_INS["ins16"], 3), (LONG_INS["ins31N"], 2)]),
             (5033, [(LONG_INS["ins12"], 2)]),
             (5026, [(COLLIDING_INSERTIONS[0][0], 2), (COLLIDING_INSERTIONS[0][1], 3)]),
             (5042, [(COLLIDING_INSERTIONS[1][1], 2), (COLLIDING_INSERTIONS[1][0], 3)]),
             (5050, [(COLLIDING_INSERTIONS[2][0], 2), (COLLIDING_INSERTIONS[2][1], 3)])]
    for anchor, alleles in sites:
        if anchor in (5026, 5042):                    # the base after the anchor is the extra base of the longer insertion
            c.set_ref("chr1", anchor + 1, "A")
    for anchor, alleles in sites:
        for ins, n_bc in alleles:
            for k in range(n_bc):
                c.both_strands("long_ins_%d" % len(ins), "chr1", anchor - 19 + k % 3, "%dM%dI20M" % (20 - k % 3, len(ins)), ins=[ins])
        for k in range(2):
            c.pair("background", "chr1", anchor - 15 + 3 * k, "40M", rev1=bool(k & 1))


GROUPS = ("cigar", "flags", "lengths", "fragments", "long_ins")


@functools.lru_cache(maxsize=None)
def build_corpus():
    c = Corpus()
    for fn in (_cigar_zoo, _flag_zoo, _read_lengths, _fragment_zoo, _long_insertions):
        fn(c)
    c.group = None
    return c


def _soa(records):
    from smcounter_b200.soa import records_to_soa
    return records_to_soa(records, [name for name, _ in CONTIGS])


def _oracle(records, intervals, refs, prm):
    index = orc.ReadIndex(records)
    rows, details = [], []
    for (chrom, pos) in loc_list(intervals):
        d = {}
        rows.append(orc.vc(index, chrom, pos, prm.minBQ, prm.minMQ, prm.mtDepth, prm.rpb, prm.hpLen, prm.mismatchThr, prm.mtDrop,
                           prm.maxMT, prm.primerDist, refs, detail=d))
        details.append(d)
    return rows, details


@functools.lru_cache(maxsize=None)
def _oracle_group(group, pname):
    c = build_corpus()
    return _oracle(c.records(group), c.intervals[group], c.refs(), PARAMS[pname])


def _detail(group, pname, chrom, pos0):
    c = build_corpus()
    k = loc_list(c.intervals[group]).index((chrom, str(pos0 + 1)))
    return _oracle_group(group, pname)[1][k]


# ---------------------------------------------------------------------------------------------- CPU: the checker itself
PILEUP_CASES = [        # (cigar, pos, column, (qpos, indel, is_del)) by htslib resolve_cigar2 (SURVEY.md A.2)
    ("5H10S40M", 100, 100, (10, 0, False)), ("5H10S40M", 100, 139, (49, 0, False)),
    ("40M10S5H", 100, 139, (39, 0, False)),
    ("3H45M4H", 100, 100, (0, 0, False)), ("3H45M4H", 100, 144, (44, 0, False)),
    ("30=1X40=", 100, 129, (29, 0, False)), ("30=1X40=", 100, 130, (30, 0, False)), ("30=1X40=", 100, 170, (70, 0, False)),
    ("20M2I15M3D20M1I10M", 100, 119, (19, 2, False)), ("20M2I15M3D20M1I10M", 100, 134, (36, -3, False)),
    ("20M2I15M3D20M1I10M", 100, 136, (37, 0, True)), ("20M2I15M3D20M1I10M", 100, 157, (56, 1, False)),
    ("20M2I15M3D20M1I10M", 100, 158, (58, 0, False)),
    ("5S3I40M", 100, 100, (8, 0, False)),
    ("40M2I6S", 100, 139, (39, 2, False)),
    ("35M4D", 100, 134, (34, -4, False)), ("35M4D", 100, 135, (35, 0, True)), ("35M4D", 100, 138, (35, 0, True)),
    ("20M2D3I20M", 100, 119, (19, -2, False)), ("20M2D3I20M", 100, 120, (20, 0, True)), ("20M2D3I20M", 100, 121, (20, 3, True)),
    ("20M2D3I20M", 100, 122, (23, 0, False)),
    ("20M3I2D20M", 100, 119, (19, 3, False)), ("20M3I2D20M", 100, 120, (23, 0, True)), ("20M3I2D20M", 100, 121, (23, 0, True)),
    ("20M3I2D20M", 100, 122, (23, 0, False)),
    ("15M40N15M", 100, 114, (14, 0, False)), ("15M40N15M", 100, 115, (15, 0, True)), ("15M40N15M", 100, 154, (15, 0, True)),
    ("15M40N15M", 100, 155, (15, 0, False)),
    ("25M2P3I25M", 100, 124, (24, 3, False)), ("25M2P3I25M", 100, 125, (28, 0, False)),
    ("25M2I1P3I25M", 100, 124, (24, 2, False)), ("25M2I1P3I25M", 100, 125, (30, 0, False)),
    ("20M6D20M", 100, 119, (19, -6, False)), ("20M6D20M", 100, 125, (20, 0, True)),
]


@pytest.mark.parametrize("cigar,pos,p,want", PILEUP_CASES)
def test_oracle_pileup_column_on_hand_derived_positions(cigar, pos, p, want):
    r = orc.Read("r:AC:1", "c", pos, 0x40, 60, 0, parse_cigar(cigar), "A" * 200, [30] * 200)
    assert pos <= p < orc.reference_end(r)
    qpos, indel, is_del = orc.pileup_column(r, p)
    assert (qpos, indel, bool(is_del)) == want


def test_reads_without_cigar_or_mapped_flag_never_pile_up():
    a = orc.Read("a:AC:1", "c", 100, 0x40, 60, 0, [], "ACGT", [30] * 4)
    b = orc.Read("b:AC:1", "c", 100, 0x44, 60, 0, [(0, 4)], "ACGT", [30] * 4)
    d = orc.Read("d:AC:1", "c", 100, 0x40, 60, 0, [(0, 4)], "ACGT", [30] * 4)
    idx = orc.ReadIndex([a, b, d])
    assert [r.qname for p in range(99, 105) for r in idx.column("c", p)] == ["d:AC:1"] * 4


def test_long_insertion_hash_collisions_are_real():
    """If this fails the device's hash changed: find new colliding pairs (same hash, one a prefix of the other plus one base,
    and one of equal length) and put them in COLLIDING_INSERTIONS, or the long-insertion cases lose their point."""
    for a, b, h in COLLIDING_INSERTIONS:
        assert a != b
        assert long_ins_hash(a) == long_ins_hash(b) == h, (a, b, hex(long_ins_hash(a)), hex(long_ins_hash(b)))
    assert len(COLLIDING_INSERTIONS[0][1]) == len(COLLIDING_INSERTIONS[0][0]) + 1 and COLLIDING_INSERTIONS[0][1].startswith(COLLIDING_INSERTIONS[0][0])
    assert len(COLLIDING_INSERTIONS[1][1]) == len(COLLIDING_INSERTIONS[1][0]) + 1 and COLLIDING_INSERTIONS[1][1].startswith(COLLIDING_INSERTIONS[1][0])
    assert len(COLLIDING_INSERTIONS[2][0]) == len(COLLIDING_INSERTIONS[2][1]) > 8


def test_corpus_is_in_bam_order_with_dense_fragment_ids():
    import numpy as np
    c = build_corpus()
    recs = c.records()
    chrom_rank = {name: k for k, (name, _) in enumerate(CONTIGS)}
    keys = [(chrom_rank[r.chrom], r.pos) for r in recs]
    assert keys == sorted(keys)
    assert all(r.flag & 0xC0 for r in recs)                  # no read is neither R1 nor R2 (a documented deviation)
    soa = _soa(recs)
    ids = soa.frag_id.astype(np.int64)
    assert set(ids.tolist()) == set(range(int(ids.max()) + 1))
    first = [int(i) for i in dict.fromkeys(ids.tolist())]
    assert first == sorted(first)                            # numbered in order of first appearance
    lens = sorted(set(int(x) for x in soa.l_seq))
    assert {1, 2, 33, 151, 300, 1000} <= set(lens)
    want = {"H_S_M", "M_S_H", "H_M_H", "eq_X", "M_eq_X_M", "multi_indel", "S_I_M", "M_I_S", "M_D_last", "D_I", "I_D", "N_skip", "M_P_I_M",
            "M_I_P_I_M", "D_across_tile", "no_cigar", "secondary", "qcfail", "duplicate", "supplementary", "unmapped", "both_r1_r2", "mapq255",
            "nm_below_indel", "mapq_at_minMQ", "bq_at_minBQ", "mm_at_threshold", "end_dist_not_plain", "len1", "len2", "len33", "len151",
            "len300", "len1000", "frag_size_1", "frag_size_2", "frag_size_3", "frag_size_4", "frag_45_reads", "barcode_with_N",
            "long_ins_9", "long_ins_12", "long_ins_16", "long_ins_17", "long_ins_18", "long_ins_10", "long_ins_31"}
    assert want <= c.cases()
    for g in GROUPS:
        assert c.records(g) and c.intervals[g]


def test_corpus_cases_show_in_the_oracle_tallies():
    """The cases mean what they say, on the checker's side: the intended alleles with their counts, the flag semantics of
    stepper='nofilter', the threshold reads on the right side of their thresholds."""
    c = build_corpus()
    ref = c.ref["chr1"]
    # long insertions: every allele, separately, with its read count
    for anchor, ins, n_reads in ((5010, LONG_INS["ins9"], 16), (5010, LONG_INS["ins16"], 12), (5010, LONG_INS["ins31N"], 8), (5033, LONG_INS["ins12"], 8),
                                 (5026, COLLIDING_INSERTIONS[0][0], 8), (5026, COLLIDING_INSERTIONS[0][1], 12),
                                 (5042, COLLIDING_INSERTIONS[1][1], 8), (5042, COLLIDING_INSERTIONS[1][0], 12),
                                 (5050, COLLIDING_INSERTIONS[2][0], 8), (5050, COLLIDING_INSERTIONS[2][1], 12)):
        for pname in PARAMS:
            d = _detail("long_ins", pname, "chr1", anchor)
            name = "INS|%s|%s" % (ref[anchor], ref[anchor] + ins)
            assert d["alleleCnt"].get(name) == n_reads, (anchor, name, d["alleleCnt"])
            assert name in d["PI"]
    assert ref[5027] == "A" and ref[5043] == "A"
    # unmapped reads: not in allMT / allFrag; both 0x40 and 0x80 set: R2 tallies
    d = _detail("flags", "p1", "chr1", 2033)
    recs = [r for r in c.records("flags") if r.pos <= 2033 < orc.reference_end(r)]
    mapped = [r for r in recs if not r.flag & 0x4]
    assert len(mapped) < len(recs)
    assert d["cvg"] == len(mapped)
    assert d["allFrag"] == len({(r.qname.split(":")[1], r.qname.split(":")[0]) for r in mapped})
    assert d["allMT"] == len({r.qname.split(":")[1] for r in mapped})
    for r in (r for r in c.records("flags") if r.flag & 0xC0 == 0xC0):
        t = {}
        p = r.pos + 5
        orc.vc(orc.ReadIndex([r]), r.chrom, str(p + 1), 20, 30, 50, 3.0, 10, 6.0, 0, 0, 2, c.refs(), detail=t)
        assert sum(t["r2Tot"].values()) == 1 and not t["r1Tot"], r
    # fragment zoo: concordant and discordant pairs, N kept, the 45-read fragment deleted and recreated
    d = _detail("fragments", "p1", "chr2", FZ_LOCUS)
    assert d["concord"].get("A", 0) > 20 and d["discord"].get("G", 0) > 3 and d["discord"].get("A", 0) > 3
    assert d["discord"].get("Y", 0) > 0 and "R" in d["alleleCnt"] and "N" in d["alleleCnt"]
    assert d["MT3"] >= 1 and d["MT10"] >= 1


# ---------------------------------------------------------------------------------------------- reference's own vc()
def _pinned(r):
    """Reads whose pileup SURVEY.md A.2 calls pysam-version independent: no N / P op, no D next to an I."""
    ops = [op for op, _ in r.cigar]
    if 3 in ops or 6 in ops:
        return False
    return not any({ops[k], ops[k + 1]} == {1, 2} for k in range(len(ops) - 1))


def test_reference_vc_on_the_pinned_corpus():
    from oracle import ref_build, ref_shims
    if not ref_build.available():
        pytest.skip("oracle/_ref not built and /root/reference absent")
    c = build_corpus()
    recs = [r for r in c.records() if _pinned(r)]
    refs = c.refs()
    ref = ref_build.load("py2")
    bam = ref_shims.register_bam("mem:hand_built.bam", recs)
    fa = ref_shims.register_fasta("mem:hand_built.fa", refs)
    index = orc.ReadIndex(recs)
    bad = []
    try:
        for pname, prm in PARAMS.items():
            args = (prm.minBQ, prm.minMQ, prm.mtDepth, prm.rpb, prm.hpLen, prm.mismatchThr, prm.mtDrop, prm.maxMT, prm.primerDist)
            for (chrom, pos) in loc_list(c.all_intervals()):
                a = orc.vc(index, chrom, pos, *args, refs)
                b = ref.vc(bam, chrom, pos, *args, fa)
                if a != b:
                    bad.append((pname, chrom, pos, a, b))
    finally:
        ref_shims.clear_registries()
    assert not bad, bad[:3]


# ---------------------------------------------------------------------------------------------- GPU
ENCODINGS = {
    "plain": lambda s, ivs: s,
    "repack": lambda s, ivs: s.repack(),
    "trim": lambda s, ivs: s.trim_to_targets(ivs),
    "trim_compact2": lambda s, ivs: s.trim_to_targets(ivs).compact(seq_bits_wanted=2),
    "trim_compact4": lambda s, ivs: s.trim_to_targets(ivs).compact(seq_bits_wanted=4),
}


def _with_env(name, value, fn):
    old = os.environ.get(name)
    os.environ[name] = value
    try:
        return fn()
    finally:
        if old is None:
            del os.environ[name]
        else:
            os.environ[name] = old


def run_group(group, pname, enc, gpu_mutate=None):
    """One group of the corpus through the CUDA path (in encoding ``enc``) and the oracle: (problems, stats)."""
    from helpers import diff_details, diff_rows, gpu_run
    c = build_corpus()
    ivs, refs = c.intervals[group], c.refs()
    o_rows, details = _oracle_group(group, pname)
    gsoa = ENCODINGS[enc](_soa(c.records(group)), ivs)
    if gpu_mutate is not None:
        gsoa = gpu_mutate(gsoa)
    g_rows, res, loci, bed_order, tm = gpu_run(gsoa, ivs, refs, PARAMS[pname])
    problems, stats = diff_details(res, loci, bed_order, details, gsoa, refs)
    problems += diff_rows(g_rows, o_rows)
    stats.update(n_dyn=tm["n_dyn"], events=tm["n_pileup_events"], pipe_chunks=tm["pipe_chunks"], scalar_bits=gsoa.scalar_bits,
                 seq_bits=gsoa.seq_bits)
    return problems, stats


@pytest.mark.gpu
@pytest.mark.parametrize("enc", sorted(ENCODINGS))
@pytest.mark.parametrize("group", GROUPS)
def test_hand_built_group_matches_oracle(group, enc):
    problems = []
    for pname in PARAMS:
        for chunks in ("1", "3"):
            p, stats = _with_env("SMC_PIPE_CHUNKS", chunks, lambda: run_group(group, pname, enc))
            print(group, enc, pname, chunks, stats)
            assert stats["events"] > 0 and stats["pipe_chunks"] == int(chunks)
            if group == "lengths" and enc.startswith("trim_compact"):
                assert stats["scalar_bits"] == 16            # reads longer than 255 bases: 16-bit scalars, unforced
            if group == "fragments" and enc.startswith("trim_compact"):
                assert stats["seq_bits"] == int(enc[-1])
            problems += ["[%s chunks=%s] %s" % (pname, chunks, x) for x in p]
    assert not problems, "\n".join(problems[:30])


@pytest.mark.gpu
def test_fragment_zoo_downsampled_by_the_product_matches_oracle_py2_sampler():
    """mtDepth small enough that ds fires at the fragment zoo's loci: the product lists the barcodes on the device (every
    fragment then takes the ordered path), draws with its own Py2 sampler and re-runs; the oracle samples independently."""
    from smcounter_b200.smCounter import call_loci
    c = build_corpus()
    ivs, refs = c.intervals["fragments"], c.refs()
    prm = VcParams(mtDepth=3, rpb=3.0, mtDrop=1, hpLen=8)
    recs = c.records("fragments")
    o_rows, details = _oracle(recs, ivs, refs, prm)
    assert sum(1 for d in details if d.get("nBC", 0) > d.get("ds", 1 << 30)) > 20
    soa = _soa(recs)
    assert call_loci(soa, ivs, refs, prm, gpus=1) == o_rows
    assert call_loci(soa.trim_to_targets(ivs).compact(), ivs, refs, prm, gpus=1) == o_rows


@pytest.mark.gpu
def test_hand_built_corpus_bam_round_trip(tmp_path):
    """The whole corpus as a BAM through smCounter.main() -- the native decoder's handling of H, =, X, N, P, unmapped records
    with a position and reads without a CIGAR, its trim test -- against the oracle's main() on the records: three files
    byte-identical.  mtDepth is high enough that no locus is down-sampled: a sample of the barcodes can leave two long
    insertions with exactly equal PI, whose order is a documented deviation (DESIGN.md section 5)."""
    from smcounter_b200 import bam, smCounter
    c = build_corpus()
    recs, refs, ivs = c.records(), c.refs(), c.all_intervals()
    soa = _soa(recs)
    fa = tmp_path / "ref.fa"
    with open(fa, "w") as fh:
        for name, n in CONTIGS:
            s = refs.fetch(name, 0, n)
            fh.write(">%s\n" % name + "".join(s[i:i + 60] + "\n" for i in range(0, n, 60)))
    bed_lines = ["%s\t%d\t%d\n" % iv for iv in ivs]
    (tmp_path / "t.bed").write_text("".join(bed_lines))
    bam.write_bam(str(tmp_path / "reads.bam"), soa, dict(CONTIGS))
    prefix = str(tmp_path / "out")
    smCounter.argParseInit()
    thr = smCounter.main({"outPrefix": prefix, "bamFile": str(tmp_path / "reads.bam"), "bedTarget": str(tmp_path / "t.bed"), "mtDepth": 50,
                          "rpb": 3.0, "refGenome": str(fa), "bedTandemRepeats": "none", "bedRepeatMaskerSubset": "none", "threshold": 8,
                          "mtDrop": 1, "hpLen": 8})
    want = orc.run(recs, bed_lines, refs, mtDepth=50, rpb=3.0, threshold=8, mtDrop=1, hpLen=8, outPrefix=prefix)
    assert thr == want[0] == 8
    for ext, body in zip((".smCounter.all.txt", ".smCounter.cut.txt", ".smCounter.cut.vcf"), want[1:]):
        assert open(prefix + ext).read() == body, ext
    called = [l.split("\t")[3] for l in want[2].splitlines()[1:]]
    assert "C" + COLLIDING_INSERTIONS[0][1] in called and "A" + COLLIDING_INSERTIONS[1][0] in called, called
