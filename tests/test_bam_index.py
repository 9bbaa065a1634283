"""Region access through a BAM index (.bai, SAMv1 section 5.2): bam.write_bam(index=True) writes the index, and read_bam with
intervals and a current .bai beside the BAM reads and inflates only the index chunks those intervals need.  Every check runs
the native decoder (smc_bam_open_indexed) and the Python one, and compares the indexed decode with the whole-file decode of
the same file field for field: the kept reads and their order, hence the fragment ids and dictionary codes, must not change."""
import os
import shutil
import struct
import zlib
from collections import namedtuple

import numpy as np
import pytest

from smcounter_b200 import bam
from smcounter_b200.soa import records_to_soa
from smcounter_b200.synth import SynthSpec, make_panel
from test_bam_io import FIELDS, _decoders

Rec = namedtuple("Rec", "qname chrom pos flag mapq nm cigar seq qual")


# ---------------------------------------------------------------------------------------------------------------- helpers
def parse_bai(data: bytes):
    """The whole .bai, pseudo-bins included: ([{bin: [(beg, end)]}, [linear]) per reference], n_no_coor or None)."""
    assert data[:4] == b"BAI\x01"
    n_ref = struct.unpack_from("<i", data, 4)[0]
    p, refs = 8, []
    for _ in range(n_ref):
        n_bin = struct.unpack_from("<i", data, p)[0]; p += 4
        bins = {}
        for _ in range(n_bin):
            b, n = struct.unpack_from("<Ii", data, p); p += 8
            bins[b] = [struct.unpack_from("<QQ", data, p + 16 * k) for k in range(n)]; p += 16 * n
        n_intv = struct.unpack_from("<i", data, p)[0]; p += 4
        refs.append((bins, list(struct.unpack_from("<%dQ" % n_intv, data, p)))); p += 8 * n_intv
    n_no_coor = struct.unpack_from("<Q", data, p)[0] if len(data) == p + 8 else None
    assert len(data) in (p, p + 8)
    return refs, n_no_coor


def spec_bin(beg, end):
    """SAMv1 section 5.3 reg2bin for [beg, end)."""
    end -= 1
    for shift, first in ((14, 4681), (17, 585), (20, 73), (23, 9), (26, 1)):
        if beg >> shift == end >> shift:
            return first + (beg >> shift)
    return 0


def ref_span(cigar, pos):
    return pos + sum(n for op, n in cigar if op in (0, 2, 3, 7, 8))


def block_offsets(path):
    """Compressed offset of every BGZF block of the file, from the BSIZE fields."""
    data = open(path, "rb").read()
    offs, off = [], 0
    while off < len(data):
        offs.append(off)
        off += struct.unpack_from("<H", data, off + 16)[0] + 1
    return offs


def walk_records(raw, first):
    """(inflated offset, end offset, refID, pos, bin, flag, cigar) of every record."""
    out, p = [], first
    while p < len(raw):
        bs, ref, pos, l_rn, _mq, b, n_cig, flag = struct.unpack_from("<iiiBBHHH", raw, p)
        cw = struct.unpack_from("<%dI" % n_cig, raw, p + 36 + l_rn)
        out.append((p, p + 4 + bs, ref, pos, b, flag, [(c & 15, c >> 4) for c in cw]))
        p += 4 + bs
    return out


def same(a, b, trim):
    assert a.n == b.n and a.chroms == b.chroms
    for f in FIELDS + (("store_lo", "store_len") if trim else ()):
        assert np.array_equal(getattr(a, f), getattr(b, f)), f
    da, db = ({k: v for k, v in x.umi_names.items() if k >> 63} for x in (a, b))       # dictionary-coded barcodes
    assert da == db
    ha, hb = a.__dict__.get("_qual_hist"), b.__dict__.get("_qual_hist")
    if ha is not None and hb is not None:
        assert np.array_equal(ha, hb)
    assert np.array_equal(np.bincount(a.qual, minlength=256), np.bincount(b.qual, minlength=256))


def decode(path, ivs, native, trim=False, threads=1):
    if native:
        return bam.read_bam(path, ivs, native=True, threads=threads, trim=trim)
    return bam.read_bam(path, ivs, native=False, trim=trim)


def check_indexed_equals_whole(path, ivs, tmp_path, trims=(False, True), threads=(1, 3, 8)):
    """``path`` has a current .bai; a copy without one is decoded as the whole file."""
    assert bam.find_index(path) == path + ".bai"
    whole = str(tmp_path / "whole_copy.bam")
    shutil.copyfile(path, whole)
    assert bam.find_index(whole) is None
    n = None
    for native in _decoders():
        for trim in trims:
            want = decode(whole, ivs, native, trim)
            for th in (threads if native else (1,)):
                got = decode(path, ivs, native, trim, th)
                same(got, want, trim)
            n = want.n
    return n


def panel_bam(tmp_path, block=1500, seed=4):
    """Three contigs with reads and one without, small BGZF blocks so that chunks span many blocks."""
    ivs = [("chr1", 1000, 1100), ("chr1", 17000, 17060), ("chr1", 140000, 140050), ("chr2", 300, 380), ("chr2", 16370, 16400),
           ("chr3", 5000, 5040), ("chr3", 200000, 200080)]
    lengths = {"chr1": 150000, "chr2": 20000, "chr3": 250000, "chrE": 10000}
    soa, refs, _ = make_panel(ivs, SynthSpec(umis_per_locus=12, rpb=2.5, indel_every=30, indel_vaf=0.2, softclip_frac=0.2), seed=seed,
                              chroms=["chr1", "chr2", "chr3", "chrE"], lengths=lengths)
    path = str(tmp_path / "panel.bam")
    bam.write_bam(path, soa, lengths, index=True, block=block)
    return path, ivs, soa


def write_raw_bam(path, raw, first, n_ref, block, empty_block_after=None):
    """Write the inflated stream ``raw`` as BGZF blocks of ``block`` bytes (plus an empty block after block number
    ``empty_block_after``) with its .bai, computed by bam.bai_bytes from the records found in ``raw``."""
    blocks = bam._bgzf_block_list(raw, 1, block)
    where = list(range(len(blocks) + 1))          # inflated bytes [k * block, (k + 1) * block) -> block number in the file
    if empty_block_after is not None:
        co = zlib.compressobj(6, zlib.DEFLATED, -15)
        c = co.compress(b"") + co.flush()
        blocks.insert(empty_block_after + 1, b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" +
                      struct.pack("<H", 25 + len(c)) + c + struct.pack("<II", 0, 0))
        where = [k if k <= empty_block_after else k + 1 for k in where]
    with open(path, "wb") as fh:
        fh.write(b"".join(blocks) + bam._BGZF_EOF)
    coff = np.concatenate(([0], np.cumsum([len(b) for b in blocks]))).tolist()
    voff = lambda p: (coff[where[p // block]] << 16) | (p % block)
    recs = [(ref, pos, max(ref_span(cig, pos), pos + 1), b, flag, s, e) for (s, e, ref, pos, b, flag, cig) in walk_records(raw, first)]
    with open(path + ".bai", "wb") as fh:
        fh.write(bam.bai_bytes(recs, n_ref, voff))


# ---------------------------------------------------------------------------------------------------------------- 1: writer
def test_index_writer_matches_the_spec_by_hand(tmp_path):
    """Six records around the 16 kbp and 128 kbp boundaries of chr1 plus an unmapped one with a position; the written .bai is
    parsed on its own and compared with bins, chunks, linear entries and pseudo-bins derived here from the specification."""
    q = lambda n: [30] * n
    recs = [Rec("r0:AC:1", "chr1", 100, 0x40, 60, 0, [(0, 50)], "A" * 50, q(50)),                  # bin 4681
            Rec("r1:AC:1", "chr1", 200, 0x40, 60, 0, [(0, 50)], "C" * 50, q(50)),                  # bin 4681 again: same chunk
            Rec("r2:AC:1", "chr1", 16360, 0x40, 60, 0, [(0, 40)], "G" * 40, q(40)),                # crosses 16384: bin 585
            Rec("r3:AC:1", "chr1", 16400, 0x40, 60, 0, [(0, 30), (2, 5), (0, 10)], "T" * 40, q(40)),  # bin 4682
            Rec("r4:AC:1", "chr1", 131000, 0x40, 60, 0, [(0, 100)], "A" * 100, q(100)),            # crosses 131072: bin 73
            Rec("r5:AC:1", "chr1", 131200, 0x44, 0, 0, [], "ACGT", q(4)),                          # unmapped, placed: bin 4689
            Rec("r6:AC:1", "chr2", 10, 0x80, 60, 0, [(4, 5), (0, 20)], "C" * 25, q(25))]           # chr2, bin 4681
    soa = records_to_soa(recs, ["chr1", "chr2", "chr3"])
    path = str(tmp_path / "hand.bam")
    block = 100
    bam.write_bam(path, soa, {"chr1": 200000, "chr2": 1000, "chr3": 500}, index=True, block=block)
    refs, n_no_coor = parse_bai(open(path + ".bai", "rb").read())
    raw = bam.bgzf_decompress(open(path, "rb").read())
    _, _, first = bam.parse_header(raw)
    walked = walk_records(raw, first)
    coff = block_offsets(path)
    voff = lambda p: (coff[p // block] << 16) | (p % block)
    beg = [voff(w[0]) for w in walked]
    end = [voff(w[1]) for w in walked]
    bins = [spec_bin(r.pos, max(ref_span(r.cigar, r.pos), r.pos + 1)) for r in recs]
    assert bins == [4681, 4681, 585, 4682, 73, 4689, 4681]
    assert [w[4] for w in walked] == bins                       # the bin each record stores
    assert len({b >> 16 for b in beg}) > 3                      # the records are spread over several blocks
    want_chr1 = {4681: [(beg[0], end[1])], 585: [(beg[2], end[2])], 4682: [(beg[3], end[3])], 73: [(beg[4], end[4])],
                 4689: [(beg[5], end[5])], 37450: [(beg[0], end[5]), (5, 1)]}
    assert refs[0][0] == want_chr1
    # linear index: the first record overlapping each 16 kbp window (r2 reaches into window 1; 0 where no record does)
    lin = [0] * 9
    lin[0], lin[1], lin[7], lin[8] = beg[0], beg[2], beg[4], beg[4]      # r4 covers [131000, 131100): windows 7 and 8
    assert refs[0][1] == lin
    assert refs[1] == ({4681: [(beg[6], end[6])], 37450: [(beg[6], end[6]), (1, 0)]}, [beg[6]])
    assert refs[2] == ({}, [])
    assert n_no_coor == 0
    # the readers agree with the test's parse
    py = bam.read_bai(path + ".bai", 3)
    assert [(bi, l) for bi, l in py] == [({k: v for k, v in r[0].items() if k != 37450}, r[1]) for r in refs]


# ---------------------------------------------------------------------------------------------------------------- 2: subsets
def _subsets(ivs):
    return {
        "one_locus": [("chr1", 1050, 1051)],
        "one_interval": [ivs[3]],
        "every_other": ivs[::2],
        "all": ivs,
        "overlapping": [("chr1", 990, 1060), ("chr1", 1040, 1110), ("chr1", 1050, 1070), ("chr3", 4990, 5100), ("chr3", 5000, 5010)],
        "contig_without_reads": [("chrE", 100, 5000)],
        "contig_not_in_bam": [("chrX", 100, 5000), ("chr2", 16380, 16390)],
        "past_contig_end": [("chr2", 19990, 400000), ("chr3", 1 << 30, (1 << 30) + 100), ("chr3", 200050, 600000000)],
    }


@pytest.mark.parametrize("subset", ["one_locus", "one_interval", "every_other", "all", "overlapping", "contig_without_reads",
                                    "contig_not_in_bam", "past_contig_end"])
def test_indexed_decode_equals_whole_file(tmp_path, subset):
    path, ivs, _ = panel_bam(tmp_path)
    n = check_indexed_equals_whole(path, _subsets(ivs)[subset], tmp_path)
    assert (n == 0) == (subset == "contig_without_reads")


def test_indexed_decode_reads_less(tmp_path):
    """One interval of seven: the chunks cover a small part of the file."""
    path, ivs, _ = panel_bam(tmp_path)
    chunks = bam.bai_chunks(bam.read_bai(path + ".bai", 4), ["chr1", "chr2", "chr3", "chrE"], [ivs[3]])
    size = os.path.getsize(path)
    assert 0 < sum((e >> 16) - (b >> 16) for b, e in chunks) < size / 3


# ---------------------------------------------------------------------------------------------------------------- 3: far reads
def test_reads_that_reach_a_target_from_far_away(tmp_path):
    q = lambda n: [20 + k % 20 for k in range(n)]
    seq = lambda n: ("ACGTTGCA" * (n // 8 + 1))[:n]
    recs, k = [], 0

    def add(pos, cigar, flag=0x40):
        nonlocal k
        n = sum(l for op, l in cigar if op in (0, 1, 4, 7, 8))
        recs.append(Rec("q%d:%s:1" % (k, "ACGTAC"[k % 3:k % 3 + 3]), "chr1", pos, flag, 60, 0, cigar, seq(n), q(n)))
        k += 1
    for p in range(0, 240000, 700):                                       # background: one read every 700 bp
        add(p, [(0, 60)])
    add(1000, [(0, 50), (3, 100000), (0, 50)])                            # N skip: second block at [101050, 101100)
    add(20000, [(0, 1000)])                                               # 1 000 bases, reaches [20990, 21000)
    add(32700, [(0, 50), (2, 200), (0, 50)])                              # deletion across 32768, ends at 33000
    add(50000, [(0, 100)])                                                # touches two targets
    recs.sort(key=lambda r: r.pos)
    soa = records_to_soa(recs, ["chr1"])
    path = str(tmp_path / "far.bam")
    bam.write_bam(path, soa, {"chr1": 300000}, index=True, block=2000)
    targets = [("chr1", 101060, 101070), ("chr1", 20990, 20995), ("chr1", 32960, 32970), ("chr1", 50010, 50020), ("chr1", 50080, 50090)]
    check_indexed_equals_whole(path, targets, tmp_path)
    for native in _decoders():
        got = bam.read_bam(path, targets, native=native)
        ends = got.ref_end()
        spans = set(zip(got.pos.tolist(), ends.tolist()))
        assert {(1000, 101100), (20000, 21000), (32700, 33000), (50000, 50100)} <= spans
        assert got.pos.tolist().count(50000) == 1


# ---------------------------------------------------------------------------------------------------------------- 4: awkward files
@pytest.mark.parametrize("case", ["multi_block_header", "records_over_many_blocks", "empty_block"])
def test_awkward_bgzf_layouts(tmp_path, case):
    path0, ivs, _ = panel_bam(tmp_path, block=0xff00)
    raw = bam.bgzf_decompress(open(path0, "rb").read())
    text, refs, first = bam.parse_header(raw)
    block, empty_after = 5000, None
    if case == "multi_block_header":                        # @CO text of 70 kB: the header spans a dozen blocks
        text = text + "".join("@CO\t%s\n" % ("comment %d " % i * 9) for i in range(700))
        head = [b"BAM\x01", struct.pack("<i", len(text)), text.encode(), struct.pack("<i", len(refs))]
        head += [struct.pack("<i", len(n) + 1) + n.encode() + b"\x00" + struct.pack("<i", l) for n, l in refs]
        head = b"".join(head)
        raw, first = head + raw[first:], len(head)
        assert first > 10 * block
    elif case == "records_over_many_blocks":
        block = 90                                          # ~300-byte records: every one spans three or more blocks
    else:
        empty_after = (len(raw) // block) // 2
    path = str(tmp_path / "awkward.bam")
    write_raw_bam(path, raw, first, len(refs), block, empty_after)
    for sub in (ivs[1:2], ivs[3:5], ivs):
        check_indexed_equals_whole(path, sub, tmp_path, threads=(1, 3))


# ---------------------------------------------------------------------------------------------------------------- 5: untouched blocks
def test_blocks_no_chunk_needs_are_never_read(tmp_path):
    path, ivs, _ = panel_bam(tmp_path, block=700)
    intact = str(tmp_path / "intact.bam")
    shutil.copyfile(path, intact)
    assert bam.find_index(intact) is None
    target = [ivs[3]]
    names = ["chr1", "chr2", "chr3", "chrE"]
    chunks = bam.bai_chunks(bam.read_bai(path + ".bai", 4), names, target)
    data = bytearray(open(path, "rb").read())
    offs = block_offsets(path)
    ends = offs[1:] + [len(data)]
    raw = bam.bgzf_decompress(bytes(data))
    first = bam.parse_header(raw)[2]
    needed = set(range(first // 700 + 1))                   # the header blocks
    for b, e in chunks:
        needed |= {k for k, o in enumerate(offs) if (b >> 16) <= o <= (e >> 16)}
    damaged = [k for k in range(len(offs)) if k not in needed]
    assert len(damaged) > 0.5 * len(offs)
    for k in damaged:
        data[offs[k]:ends[k]] = b"\xa5" * (ends[k] - offs[k])
    with open(path, "wb") as fh:
        fh.write(bytes(data))
    os.utime(path + ".bai")                                 # the index stays current
    damaged_copy = str(tmp_path / "damaged_no_index.bam")
    shutil.copyfile(path, damaged_copy)
    for native in _decoders():
        for trim in (False, True):
            want = decode(intact, target, native, trim, 3)           # the intact copy has no index: the whole file
            got = decode(path, target, native, trim, 3)
            assert want.n > 0
            same(got, want, trim)
        with pytest.raises(ValueError):
            decode(damaged_copy, target, native)


# ---------------------------------------------------------------------------------------------------------------- 6: selection
def test_stale_index_gives_a_warning_and_the_whole_file(tmp_path, capsys):
    path, ivs, _ = panel_bam(tmp_path)
    t = os.path.getmtime(path)
    os.utime(path + ".bai", (t - 100, t - 100))
    capsys.readouterr()
    assert bam.find_index(path) is None
    assert "older than" in capsys.readouterr().out
    for native in _decoders():
        got = bam.read_bam(path, [ivs[0]], native=native)
        out = capsys.readouterr().out
        assert out.count("warning: BAM index %s.bai is older than" % path) == 1
        shutil.move(path + ".bai", path + ".hidden")
        same(got, bam.read_bam(path, [ivs[0]], native=native), False)
        shutil.move(path + ".hidden", path + ".bai")
        os.utime(path + ".bai", (t - 100, t - 100))


def test_index_names_and_csi(tmp_path):
    path, ivs, _ = panel_bam(tmp_path)
    stem = path[:-4] + ".bai"
    shutil.move(path + ".bai", stem)
    assert bam.find_index(path) == stem
    whole = str(tmp_path / "whole_copy.bam")
    shutil.copyfile(path, whole)
    for native in _decoders():
        same(decode(path, [ivs[2]], native, True, 2), decode(whole, [ivs[2]], native, True, 2), True)
    shutil.move(stem, path + ".csi")                        # a .csi is not read: the whole-file path
    assert bam.find_index(path) is None
    for native in _decoders():
        assert bam.read_bam(path, [ivs[2]], native=native).n > 0


def _bad_indexes(path):
    good = open(path + ".bai", "rb").read()
    yield "bad_magic", b"CSI\x01" + good[4:], "bad magic"
    yield "n_ref", good[:4] + struct.pack("<i", 3) + good[8:], "n_ref"
    yield "truncated", good[:len(good) - 30], "truncated"
    yield "empty", b"", "bad magic"


@pytest.mark.parametrize("what", ["bad_magic", "n_ref", "truncated", "empty"])
def test_malformed_index_raises_naming_it(tmp_path, what):
    path, ivs, _ = panel_bam(tmp_path)
    data, msg = {k: (d, m) for k, d, m in _bad_indexes(path)}[what]
    with open(path + ".bai", "wb") as fh:
        fh.write(data)
    for native in _decoders():
        with pytest.raises(IOError, match=msg) as ei:
            bam.read_bam(path, [ivs[0]], native=native)
        assert path + ".bai" in str(ei.value)
    assert bam.read_bam(path, None).n > 0                    # without intervals the index is not used


@pytest.mark.parametrize("shift", ["past_end", "not_bgzf"])
def test_index_pointing_off_the_blocks_raises_naming_it(tmp_path, shift):
    """Chunks whose compressed offsets lie past the end of the file or inside a block: an error naming the index, never a
    silent loss of reads."""
    path, ivs, _ = panel_bam(tmp_path)
    refs, n_no_coor = parse_bai(open(path + ".bai", "rb").read())
    size = os.path.getsize(path)
    move = (lambda v: v + ((size + 10) << 16)) if shift == "past_end" else (lambda v: v + (3 << 16))
    out = [b"BAI\x01", struct.pack("<i", len(refs))]
    for bins, lin in refs:
        out.append(struct.pack("<i", len(bins)))
        for b, ch in bins.items():
            ch = ch if b == 37450 else [(move(x), move(y)) for x, y in ch]
            out.append(struct.pack("<Ii", b, len(ch)) + b"".join(struct.pack("<QQ", x, y) for x, y in ch))
        out.append(struct.pack("<i", len(lin)) + b"".join(struct.pack("<Q", x) for x in lin))
    out.append(struct.pack("<Q", n_no_coor))
    with open(path + ".bai", "wb") as fh:
        fh.write(b"".join(out))
    for native in _decoders():
        with pytest.raises(IOError, match="past the end" if shift == "past_end" else "BGZF") as ei:
            bam.read_bam(path, [ivs[0]], native=native, threads=2)
        assert path + ".bai" in str(ei.value)


# ---------------------------------------------------------------------------------------------------------------- 7: hand-built corpus
def test_hand_built_corpus_indexed_equals_whole_file(tmp_path):
    """H / N / P CIGARs, reads without a CIGAR, unmapped records with a position (tests/test_gpu_hand_built_reads.py)."""
    from test_gpu_hand_built_reads import CONTIGS, _soa, build_corpus
    c = build_corpus()
    soa = _soa(c.records())
    path = str(tmp_path / "corpus.bam")
    bam.write_bam(path, soa, dict(CONTIGS), index=True, block=1000)
    ivs = c.all_intervals()
    check_indexed_equals_whole(path, ivs, tmp_path)
    check_indexed_equals_whole(path, ivs[::3], tmp_path, threads=(1, 4))


# ---------------------------------------------------------------------------------------------------------------- 8: shared boundary
def test_reads_without_reference_length_at_a_boundary_two_intervals_share(tmp_path):
    """Mapped reads that consume no reference (CIGAR 10S, no CIGAR) around [1000, 1100) and [1100, 1200).  Such a read at p
    touches an interval only when start < p < end, so the ones at 1000, 1100 and 1200 are dropped: the two intervals must not
    act as one [1000, 1200).  The native decoder, whole file and indexed, equals the Python one, trimmed and untrimmed."""
    q = lambda n: [30 + k % 7 for k in range(n)]
    recs = []

    def add(pos, cigar, n):
        recs.append(Rec("r%d:ACGT:1" % len(recs), "chr1", pos, 0x40, 60, 0, cigar, ("ACGTTGCA" * 8)[:n], q(n)))
    for p in (999, 1000, 1001, 1099, 1100, 1101, 1199, 1200, 1201):
        add(p, [(4, 10)], 10)
        add(p, [], 12)
    add(1080, [(4, 3), (0, 40), (4, 2)], 45)                  # aligned across the shared boundary: trimmed to [1080, 1120)
    add(1190, [(0, 30)], 30)
    recs.sort(key=lambda r: r.pos)
    soa = records_to_soa(recs, ["chr1"])
    path = str(tmp_path / "edge.bam")
    bam.write_bam(path, soa, {"chr1": 5000}, index=True, block=200)
    whole = str(tmp_path / "edge_whole.bam")
    shutil.copyfile(path, whole)
    ivs = [("chr1", 1000, 1100), ("chr1", 1100, 1200)]
    for trim in (False, True):
        want = decode(whole, ivs, False, trim)
        no_span = want.pos[want.ref_end() == want.pos].tolist()
        assert no_span == [1001, 1001, 1099, 1099, 1101, 1101, 1199, 1199]
        assert want.n == len(no_span) + 2
        if len(_decoders()) > 1:
            for p in (whole, path):
                for th in (1, 3):
                    same(decode(p, ivs, True, trim, th), want, trim)


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_cli_output_identical_with_and_without_the_index(tmp_path):
    """smCounter.main() on a multi-contig BAM whose BED covers about a tenth of its intervals, once without and once with the
    .bai: the three files are byte-identical."""
    from smcounter_b200 import _bamio, smCounter
    ivs = [("chr%d" % (1 + k % 3), 2000 + 6000 * (k // 3), 2000 + 6000 * (k // 3) + 60) for k in range(30)]
    soa, refs, _ = make_panel(ivs, SynthSpec(umis_per_locus=30, rpb=3.0, snv_every=25, snv_vaf=0.2, indel_every=40, indel_vaf=0.15), seed=77)
    fa = tmp_path / "ref.fa"
    with open(fa, "w") as fh:
        for ch in soa.chroms:
            s = refs.fetch(ch, 0, refs.get_reference_length(ch))
            fh.write(">%s\n" % ch + "".join(s[i:i + 60] + "\n" for i in range(0, len(s), 60)))
    sub = ivs[::10]
    (tmp_path / "t.bed").write_text("".join("%s\t%d\t%d\n" % iv for iv in sub))
    path = str(tmp_path / "reads.bam")
    bam.write_bam(path, soa, refs.lengths, index=True, block=4000)
    used = []
    orig = _bamio.read_bam_native

    def spy(*a, **kw):
        used.append(kw.get("index"))
        return orig(*a, **kw)
    smCounter.argParseInit()
    args = {"bamFile": path, "bedTarget": str(tmp_path / "t.bed"), "mtDepth": 60, "rpb": 3.0, "refGenome": str(fa),
            "bedTandemRepeats": "none", "bedRepeatMaskerSubset": "none", "threshold": 10}
    prefix = str(tmp_path / "out")                       # one prefix for both runs: it names the VCF's sample column
    exts = (".smCounter.all.txt", ".smCounter.cut.txt", ".smCounter.cut.vcf")
    _bamio.read_bam_native = spy
    try:
        shutil.move(path + ".bai", path + ".hidden")
        smCounter.main(dict(args, outPrefix=prefix))
        whole = [open(prefix + ext, "rb").read() for ext in exts]
        shutil.move(path + ".hidden", path + ".bai")
        smCounter.main(dict(args, outPrefix=prefix))
        indexed = [open(prefix + ext, "rb").read() for ext in exts]
    finally:
        _bamio.read_bam_native = orig
    assert used == [None, path + ".bai"]
    for ext, a, b in zip(exts, whole, indexed):
        assert a == b, ext
    assert len(whole[0].splitlines()) > 150


@pytest.mark.gpu
def test_hand_built_corpus_bam_round_trip_through_the_index(tmp_path):
    """The hand-built corpus round trip (oracle main() against product main(), three files byte-identical) on an indexed BAM."""
    from oracle import smcounter_oracle as orc
    from smcounter_b200 import _bamio, smCounter
    from test_gpu_hand_built_reads import CONTIGS, _soa, build_corpus
    c = build_corpus()
    recs, refs, ivs = c.records(), c.refs(), c.all_intervals()
    fa = tmp_path / "ref.fa"
    with open(fa, "w") as fh:
        for name, n in CONTIGS:
            s = refs.fetch(name, 0, n)
            fh.write(">%s\n" % name + "".join(s[i:i + 60] + "\n" for i in range(0, n, 60)))
    bed_lines = ["%s\t%d\t%d\n" % iv for iv in ivs]
    (tmp_path / "t.bed").write_text("".join(bed_lines))
    path = str(tmp_path / "reads.bam")
    bam.write_bam(path, _soa(recs), dict(CONTIGS), index=True, block=1000)
    prefix = str(tmp_path / "out")
    used = []
    orig = _bamio.read_bam_native

    def spy(*a, **kw):
        used.append(kw.get("index"))
        return orig(*a, **kw)
    smCounter.argParseInit()
    _bamio.read_bam_native = spy
    try:
        thr = smCounter.main({"outPrefix": prefix, "bamFile": path, "bedTarget": str(tmp_path / "t.bed"), "mtDepth": 50, "rpb": 3.0,
                              "refGenome": str(fa), "bedTandemRepeats": "none", "bedRepeatMaskerSubset": "none", "threshold": 8,
                              "mtDrop": 1, "hpLen": 8})
    finally:
        _bamio.read_bam_native = orig
    assert used == [path + ".bai"]
    want = orc.run(recs, bed_lines, refs, mtDepth=50, rpb=3.0, threshold=8, mtDrop=1, hpLen=8, outPrefix=prefix)
    assert thr == want[0] == 8
    for ext, body in zip((".smCounter.all.txt", ".smCounter.cut.txt", ".smCounter.cut.vcf"), want[1:]):
        assert open(prefix + ext).read() == body, ext
