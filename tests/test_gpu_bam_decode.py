"""BAM decode on the GPU (include/smc_b200.h: smc_decode_bam, bam.read_bam(..., device=0)): the device inflater against zlib
and the host routine, and the decoded arrays against the host decoder's, element for element, on every kind of file the host
decoder's tests use; the CLI with --bamDecoder gpu writes the same files as with the host decoder."""
import ctypes as C
import os
import struct
import zlib

import numpy as np
import pytest

from smcounter_b200 import bam
from smcounter_b200.synth import SynthSpec, make_panel

pytestmark = pytest.mark.gpu

FIELDS = ("ref_id", "pos", "flag", "mapq", "nm", "l_seq", "seq_off", "qual_off", "cigar_off", "n_cigar", "umi", "frag_id", "seq",
          "qual", "cigar")


def _panel(seed=2, **kw):
    spec = SynthSpec(**dict(dict(umis_per_locus=15, rpb=2.5, snv_every=30, snv_vaf=0.2, indel_every=40, indel_vaf=0.2, softclip_frac=0.2), **kw))
    ivs = [("chr1", 400, 460), ("chr2", 150, 170)]
    s, refs, _ = make_panel(ivs, spec, seed=seed)
    return s, refs, ivs


def _same(path, intervals=None, trim=False):
    """read_bam on the GPU equals the host decoder, and the GPU did decode it"""
    want = bam.read_bam(path, intervals, native=True, trim=trim)
    got = bam.read_bam(path, intervals, trim=trim, device=0)
    assert got.__dict__.get("_bam_decoder") == "device"
    assert got.n == want.n and got.chroms == want.chroms and got.packed
    for f in FIELDS + ("store_lo", "store_len"):
        a, b = getattr(got, f), getattr(want, f)
        assert (a is None) == (b is None), f
        assert a is None or (a.dtype == b.dtype and np.array_equal(a, b)), f
    assert got.umi_names == want.umi_names
    assert np.array_equal(got.__dict__["_qual_hist"], want.__dict__["_qual_hist"])
    return got


# ---------------------------------------------------------------------------------------------------------------- inflate
def _device_inflate(streams):
    """[(compressed, out_len)] through smc_inflate_device: (status, outputs); a canary after every output slice"""
    from smcounter_b200 import _ffi
    fl = _ffi.load()
    ctx = C.c_void_p()
    assert fl.smc_ctx_create(0, C.byref(_ffi.smc_params()), C.byref(ctx)) == 0
    try:
        in_off, in_len, out_off, out_len, ib, ob = [], [], [], [], 0, 0
        for comp, n in streams:
            in_off.append(ib); in_len.append(len(comp)); ib += len(comp) + 64
            out_off.append(ob); out_len.append(n); ob += n + 64
        src = np.zeros(max(ib, 1), np.uint8)
        for (comp, _), o in zip(streams, in_off):
            src[o:o + len(comp)] = np.frombuffer(comp, np.uint8)
        dst = np.full(max(ob, 1), 0xAB, np.uint8)
        st = np.zeros(len(streams), np.int32)
        a = lambda v: np.asarray(v, np.int64)
        io, il, oo, ol = a(in_off), a(in_len), a(out_off), a(out_len)
        rc = fl.smc_inflate_device(ctx, len(streams), src.ctypes.data, len(src), io.ctypes.data, il.ctypes.data, dst.ctypes.data, len(dst),
                                   oo.ctypes.data, ol.ctypes.data, st.ctypes.data)
        assert rc == 0, fl.smc_last_error(ctx)
        for o, n in zip(out_off, out_len):
            assert (dst[o + n:o + n + 64] == 0xAB).all(), "wrote past the output"
        return st, [dst[o:o + n].tobytes() for o, n in zip(out_off, out_len)]
    finally:
        fl.smc_ctx_destroy(ctx)


def test_device_inflate_equals_zlib_on_every_kind_of_stream():
    """The corpus of the host routine's test (random bytes of several entropies, text, BAM records, runs, empty input; levels
    0/1/4/6/9 with the default, fixed, Huffman-only, RLE and filtered strategies; several deflate blocks in one stream):
    zlib's bytes, nothing written past any output."""
    rng = np.random.default_rng(12)
    data_sets = [b"", b"a", b"ab" * 7]
    for n in (1, 2, 7, 8, 9, 15, 16, 17, 255, 256, 257, 258, 259, 4095, 65280):
        data_sets += [bytes(rng.integers(0, 256, size=n, dtype=np.uint8)), bytes(rng.integers(0, 4, size=n, dtype=np.uint8)),
                      (b"ACGT" * (n // 4 + 1))[:n], b"\x00" * n, bytes(np.repeat(rng.integers(0, 256, size=n // 9 + 1, dtype=np.uint8), 9)[:n])]
    data_sets.append((b"the quick brown fox jumps over the lazy dog. " * 900)[:40000])
    s, refs, _ = _panel(seed=3)
    p = "/tmp/_smc_dev_inflate_case.bam"
    bam.write_bam(p, s, refs.lengths)
    data_sets.append(bam.bgzf_decompress(open(p, "rb").read())[:65280])
    os.remove(p)
    data_sets.append(bytes(rng.integers(0, 256, size=20000, dtype=np.uint8)) + b"\x07" * 20000 + bytes(rng.integers(0, 16, size=20000, dtype=np.uint8)))
    streams, want = [], []
    for data in data_sets:
        for level in (0, 1, 4, 6, 9):
            for strategy in (zlib.Z_DEFAULT_STRATEGY, zlib.Z_FIXED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FILTERED):
                co = zlib.compressobj(level, zlib.DEFLATED, -15, 9, strategy)
                streams.append((co.compress(data) + co.flush(), len(data))); want.append(data)
        co = zlib.compressobj(6, zlib.DEFLATED, -15)
        half = len(data) // 2
        streams.append((co.compress(data[:half]) + co.flush(zlib.Z_FULL_FLUSH) + co.compress(data[half:]) + co.flush(), len(data)))
        want.append(data)
    st, got = _device_inflate(streams)
    assert (st == 0).all()
    for g, w in zip(got, want):
        assert g == w
    assert len(streams) > 1500


def test_device_inflate_on_hand_made_dynamic_blocks():
    """The streams of test_own_inflate_on_hand_made_dynamic_blocks (same generator, same seed): dynamic-Huffman blocks with random
    complete codes of up to 15 bits on both alphabets (the decoder's secondary tables) and single-code distance alphabets (the
    incomplete code RFC 1951 allows), every length / distance symbol with its extra bits.  zlib's bytes on the device."""
    from test_bam_io import _BitWriter, _canonical_codes, _random_code_lengths
    LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
    LEN_EXTRA = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
    DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577]
    DIST_EXTRA = [0, 0, 0, 0] + [k for k in range(1, 14) for _ in (0, 1)]
    ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
    rng = np.random.default_rng(31)
    deepest, n_single, streams, want = 0, 0, [], []
    for case in range(120):
        deep = case % 2 == 0
        n_lit = int(rng.integers(2, 286))
        lit_lens = _random_code_lengths(rng, n_lit, 286, must_have=(256,), deep=deep)
        n_dist = int(rng.integers(1, 31))
        dist_lens = _random_code_lengths(rng, n_dist, 30, deep=deep) if n_dist > 1 else [0] * 30
        if n_dist == 1:
            dist_lens[int(rng.integers(0, 30))] = 1
            n_single += 1
        deepest = max(deepest, max(lit_lens), max(dist_lens))
        lit_codes, dist_codes = _canonical_codes(lit_lens), _canonical_codes(dist_lens)
        pre_lens = [0] * 19
        for k, s in enumerate(rng.permutation(19)):
            pre_lens[int(s)] = 4 if k < 13 else 5
        pre_codes = _canonical_codes(pre_lens)
        w = _BitWriter()
        w.bits(1, 1); w.bits(2, 2)
        w.bits(286 - 257, 5); w.bits(30 - 1, 5); w.bits(19 - 4, 4)
        for s in ORDER:
            w.bits(pre_lens[s], 3)
        for l in lit_lens + dist_lens:
            w.code(pre_codes[l])
        out = bytearray()
        lits = [s for s in lit_codes if s < 256]
        lens_syms = [s for s in lit_codes if s > 256]
        dsyms = list(dist_codes)
        for step in range(int(rng.integers(1, 400))):
            can_match = lens_syms and len(out) > 0 and any(DIST_BASE[d] <= len(out) for d in dsyms)
            if lits and (not can_match or rng.random() < 0.5):
                s = int(rng.choice(lits))
                w.code(lit_codes[s]); out.append(s)
            elif can_match:
                ls = int(rng.choice(lens_syms))
                ds = int(rng.choice([d for d in dsyms if DIST_BASE[d] <= len(out)]))
                le = int(rng.integers(0, 1 << LEN_EXTRA[ls - 257])) if LEN_EXTRA[ls - 257] else 0
                dmax = min((1 << DIST_EXTRA[ds]) - 1, len(out) - DIST_BASE[ds])
                de = int(rng.integers(0, dmax + 1))
                length, dist = LEN_BASE[ls - 257] + le, DIST_BASE[ds] + de
                w.code(lit_codes[ls]); w.bits(le, LEN_EXTRA[ls - 257])
                w.code(dist_codes[ds]); w.bits(de, DIST_EXTRA[ds])
                for _ in range(length):
                    out.append(out[-dist])
        w.code(lit_codes[256])
        stream = w.done()
        assert zlib.decompress(stream, -15) == bytes(out), "the test's encoder is wrong"
        streams.append((stream, len(out))); want.append(bytes(out))
    st, got = _device_inflate(streams)
    assert (st == 0).all()
    for k, (g, w_) in enumerate(zip(got, want)):
        assert g == w_, k
    assert deepest == 15 and n_single > 0


def test_device_inflate_rejects_what_the_host_routine_rejects():
    """Wrong sizes, truncations, flipped bits and garbage: the device returns -1 exactly where smc_bam_inflate_raw does, and the
    same bytes where both accept; nothing is written past an output."""
    import test_bam_io as T
    rng = np.random.default_rng(5)
    data = bytes(rng.integers(0, 8, size=30000, dtype=np.uint8)) + b"GATTACA" * 500
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    comp = co.compress(data) + co.flush()
    cases = [(comp, len(data)), (comp, len(data) - 1), (comp, len(data) + 1)] + [(comp[:c], len(data)) for c in (1, 2, 10, len(comp) // 2, len(comp) - 1)]
    for _ in range(400):
        b = bytearray(comp)
        b[int(rng.integers(0, len(b)))] ^= 1 << int(rng.integers(0, 8))
        cases.append((bytes(b), len(data)))
    for _ in range(200):
        cases.append((bytes(rng.integers(0, 256, size=int(rng.integers(1, 400)), dtype=np.uint8)), 1000))
    st, got = _device_inflate(cases)
    n_bad = 0
    for (c, n), s, g in zip(cases, st, got):
        rc, h = T._native_inflate(c, n)
        assert s == rc
        if rc == 0:
            assert g == h
        n_bad += rc != 0
    assert n_bad > 300


# ---------------------------------------------------------------------------------------------------------------- decode
@pytest.mark.parametrize("block", [512, 4099, 0xff00])
def test_panel_whole_file_and_indexed(tmp_path, block):
    """Synthetic panel, BGZF blocks of 512 bytes and up (records cut across two or more blocks): whole file, through the .bai,
    trim on and off, no intervals, intervals that match nothing"""
    s, refs, ivs = _panel(seed=5)
    path = str(tmp_path / "t.bam")
    bam.write_bam(path, s, refs.lengths, index=True, block=block)
    _same(path)
    for trim in (False, True):
        got = _same(path, ivs, trim)                       # through the index
        assert got.n > 0
    _same(path, [("chr1", 100000, 100100)])
    _same(path, [("chrX", 1, 100)])
    os.remove(path + ".bai")
    for trim in (False, True):
        _same(path, ivs, trim)                             # whole file with intervals


def test_long_reads_small_blocks(tmp_path):
    """Reads of 1 000 bases in 512-byte blocks: every record spans several blocks, some ranges hold no record start"""
    spec = SynthSpec(umis_per_locus=6, rpb=2.0, read_len=1000, spacing=1000, frag_extra=50, snv_every=100, snv_vaf=0.2)
    ivs = [("chr1", 3000, 3100)]
    s, refs, _ = make_panel(ivs, spec, seed=4)
    path = str(tmp_path / "long.bam")
    bam.write_bam(path, s, refs.lengths, index=True, block=512)
    _same(path)
    _same(path, ivs, True)


def test_streams_as_other_writers_make_them(tmp_path):
    """Irregular blocks that cut records and the block_size field, every deflate flavour, extra gzip subfields, an empty block
    in the middle, the EOF marker (the streams of test_bgzf_streams_as_other_writers_make_them)"""
    s, refs, ivs = _panel(seed=11)
    path = str(tmp_path / "a.bam")
    bam.write_bam(path, s, refs.lengths)
    raw = bam.bgzf_decompress(open(path, "rb").read())
    rng = np.random.default_rng(7)
    flavours = [(0, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_FIXED), (1, zlib.Z_DEFAULT_STRATEGY), (9, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_HUFFMAN_ONLY)]

    def block(chunk, level, strategy, extra_subfield):
        co = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
        c = co.compress(chunk) + co.flush()
        extra = (b"XY\x03\x00abc" if extra_subfield else b"") + b"BC\x02\x00"
        xlen = len(extra) + 2
        bsize = 12 + xlen + len(c) + 8 - 1
        return (b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff" + struct.pack("<H", xlen) + extra + struct.pack("<H", bsize) + c +
                struct.pack("<II", zlib.crc32(chunk) & 0xffffffff, len(chunk)))
    out, p, k = [], 0, 0
    while p < len(raw):
        n = int(rng.choice([1, 3, 37, 501, 4099, 30011]))
        level, strategy = flavours[k % len(flavours)]
        out.append(block(raw[p:p + n], level, strategy, k % 3 == 1))
        if k == 5:
            out.append(block(b"", 6, zlib.Z_DEFAULT_STRATEGY, False))
        p += n
        k += 1
    out.append(bam._BGZF_EOF)
    path2 = str(tmp_path / "b.bam")
    with open(path2, "wb") as fh:
        fh.write(b"".join(out))
    _same(path2)
    _same(path2, ivs, True)


@pytest.mark.parametrize("nm_type", ["c", "C", "s", "S", "i", "I"])
def test_tags_nm_types_and_unmapped(tmp_path, nm_type):
    """NM of every integer type after tags of type A/c/S/f/B/Z/H, unmapped records, and files without NM"""
    s, refs, ivs = _panel(seed=8)
    s.flag = s.flag.copy()
    s.flag[3] |= 0x4
    s.flag[10] |= 0x4
    extra = b"RGZgrp1\x00" + b"XAc\xff" + b"XBS\x01\x02" + b"XCf\x00\x00\x80\x3f" + b"XDBc\x03\x00\x00\x00\x01\x02\x03" + b"XEH1AE3\x00"
    path = str(tmp_path / "t.bam")
    bam.write_bam(path, s, refs.lengths, nm_type=nm_type, extra_tags=extra)
    _same(path)
    _same(path, ivs, True)
    raw = bam.bgzf_decompress(open(path, "rb").read())
    _, _, first = bam.parse_header(raw)
    parts, p = [raw[:first]], first
    while p < len(raw):                                   # strip NM from every record
        bs = struct.unpack_from("<i", raw, p)[0]
        body = raw[p + 4:p + 4 + bs]
        body = body[:body.rindex(b"NM" + nm_type.encode())]
        parts.append(struct.pack("<i", len(body)) + body)
        p += 4 + bs
    nonm = str(tmp_path / "nonm.bam")
    with open(nonm, "wb") as fh:
        fh.write(bam.bgzf_compress(b"".join(parts), block=3000))
    assert (_same(nonm).nm == 0).all()


def test_qnames_with_any_number_of_colons_and_dictionary_barcodes(tmp_path):
    """Read names with 0, 1, 2 and many ':'; barcodes that need the dictionary (non-ACGT, longer than 31 nt) and their strings"""
    s, refs, ivs = _panel(seed=17)
    odd = {3: "ACGTNACGTACG", 11: "A" * 40, 12: "ACGTNACGTACG", 30: "TTTTGGGGNNNN"}
    shapes = [lambda fid, bc: "R%d" % fid, lambda fid, bc: "R%d:%s" % (fid, bc), lambda fid, bc: "%s:R%d" % (bc, fid),
              lambda fid, bc: "A:B:C:D:%d:%s:%d" % (fid, bc, 1), lambda fid, bc: "::%s:" % bc]
    for k, shape in enumerate(shapes):
        path = str(tmp_path / ("q%d.bam" % k))
        bam.write_bam(path, s, refs.lengths, qname_fn=lambda i, fid, bc: shape(fid, odd.get(i % 40, bc)), block=2000)
        got = _same(path)
        _same(path, ivs, True)
        if k == 3:
            assert got.umi_names and any(v == "A" * 40 for v in got.umi_names.values())


def test_hand_built_corpus(tmp_path):
    """The hand-built reads of test_gpu_hand_built_reads (H, =, X, N, P, unmapped records, long insertions)"""
    from test_gpu_hand_built_reads import CONTIGS, _soa, build_corpus
    c = build_corpus()
    path = str(tmp_path / "hand.bam")
    bam.write_bam(path, _soa(c.records()), dict(CONTIGS), index=True, block=1000)
    _same(path)
    for trim in (False, True):
        _same(path, c.all_intervals(), trim)


def test_malformed_records_raise_like_the_host(tmp_path):
    """A stream cut inside a record and a record whose fields exceed its block_size: the host path's exception type and
    message; the process (and the GPU) stay usable"""
    s, refs, ivs = _panel(seed=12)
    path = str(tmp_path / "t.bam")
    bam.write_bam(path, s, refs.lengths)
    raw = bam.bgzf_decompress(open(path, "rb").read())
    cut = str(tmp_path / "cut.bam")
    with open(cut, "wb") as fh:
        fh.write(bam.bgzf_compress(raw[:len(raw) - 1000], 1, block=3000))
    with pytest.raises(ValueError) as host_err:
        bam.read_bam(cut, native=True)
    with pytest.raises(ValueError) as dev_err:
        bam.read_bam(cut, device=0)
    assert str(dev_err.value) == str(host_err.value) and "truncated BAM record at offset" in str(dev_err.value)
    _, _, first = bam.parse_header(raw)
    bad = bytearray(raw)
    p = first
    for _ in range(7):
        p += 4 + struct.unpack_from("<i", raw, p)[0]
    struct.pack_into("<i", bad, p + 4 + 16, 100000)          # l_seq of the 8th record far beyond its block_size
    mal = str(tmp_path / "mal.bam")
    with open(mal, "wb") as fh:
        fh.write(bam.bgzf_compress(bytes(bad)))
    with pytest.raises(ValueError) as host_err:
        bam.read_bam(mal, native=True)
    with pytest.raises(ValueError) as dev_err:
        bam.read_bam(mal, device=0)
    assert str(dev_err.value) == str(host_err.value)
    _same(path)


def test_stream_over_the_device_budget_falls_back_to_the_host(tmp_path, monkeypatch, capsys):
    s, refs, ivs = _panel(seed=6)
    path = str(tmp_path / "t.bam")
    bam.write_bam(path, s, refs.lengths)
    monkeypatch.setenv("SMC_BAM_DEVICE_BUDGET", "1000")
    got = bam.read_bam(path, device=0)
    assert got.__dict__["_bam_decoder"] == "host"
    assert "exceeds the device budget" in capsys.readouterr().out
    want = bam.read_bam(path, native=True)
    for f in FIELDS:
        assert np.array_equal(getattr(got, f), getattr(want, f)), f


def test_block_the_device_inflater_rejects_falls_back_to_the_host(tmp_path, capsys):
    """A BGZF block the device inflater rejects (here: a deflate block of the reserved type, which zlib rejects as well): the
    decode goes to the host with a warning naming the block, and the host's own verdict stands"""
    s, refs, ivs = _panel(seed=9)
    path = str(tmp_path / "t.bam")
    bam.write_bam(path, s, refs.lengths, block=3000)
    data = bytearray(open(path, "rb").read())
    second = struct.unpack_from("<H", data, 16)[0] + 1            # offset of the second block (BSIZE + 1 of the first)
    data[second + 18] = 0x07                                       # BFINAL = 1, BTYPE = 11 (reserved)
    bad = str(tmp_path / "bad.bam")
    open(bad, "wb").write(bytes(data))
    with pytest.raises(ValueError) as host_err:
        bam.read_bam(bad, native=True)
    with pytest.raises(ValueError) as dev_err:
        bam.read_bam(bad, device=0)
    assert "the device inflater rejects BGZF block 1" in capsys.readouterr().out
    assert str(dev_err.value) == str(host_err.value)
    _same(path)


# ---------------------------------------------------------------------------------------------------------------- CLI
def _cli_files(tmp_path, path, fa, bed, decoder, extra):
    from smcounter_b200 import smCounter
    smCounter.argParseInit()
    prefix = str(tmp_path / "out")
    smCounter.main(dict(dict(outPrefix=prefix, bamFile=path, bedTarget=bed, refGenome=str(fa), bedTandemRepeats="none",
                             bedRepeatMaskerSubset="none", bamDecoder=decoder), **extra))
    return [open(prefix + ext, "rb").read() for ext in (".smCounter.all.txt", ".smCounter.cut.txt", ".smCounter.cut.vcf")]


def _fasta(tmp_path, names, refs):
    fa = tmp_path / "ref.fa"
    with open(fa, "w") as fh:
        for ch in names:
            s = refs.fetch(ch, 0, refs.get_reference_length(ch))
            fh.write(">%s\n" % ch + "".join(s[i:i + 60] + "\n" for i in range(0, len(s), 60)))
    return fa


def test_identities_sharing_one_name(tmp_path):
    """Read names without ':' (barcode and readid empty): every kept read is one fragment of one barcode, a single run of equal
    identity hashes as long as the file"""
    s, refs, ivs = _panel(seed=13)
    path = str(tmp_path / "t.bam")
    bam.write_bam(path, s, refs.lengths, qname_fn=lambda i, fid, bc: "R", block=5000)
    got = _same(path)
    assert got.n > 100 and (got.frag_id == 0).all()


def test_cli_gpu_decoder_writes_the_same_files(tmp_path):
    ivs = [("chr%d" % (1 + k % 3), 2000 + 6000 * (k // 3), 2000 + 6000 * (k // 3) + 60) for k in range(30)]
    soa, refs, _ = make_panel(ivs, SynthSpec(umis_per_locus=30, rpb=3.0, snv_every=25, snv_vaf=0.2, indel_every=40, indel_vaf=0.15), seed=77)
    fa = _fasta(tmp_path, soa.chroms, refs)
    bed = tmp_path / "t.bed"
    bed.write_text("".join("%s\t%d\t%d\n" % iv for iv in ivs[::3]))
    path = str(tmp_path / "reads.bam")
    bam.write_bam(path, soa, refs.lengths, index=True, block=4000)
    extra = dict(mtDepth=60, rpb=3.0, threshold=10)
    host = _cli_files(tmp_path, path, fa, str(bed), "host", extra)
    gpu = _cli_files(tmp_path, path, fa, str(bed), "gpu", extra)
    assert host == gpu and len(host[0].splitlines()) > 100


def test_cli_gpu_decoder_on_the_hand_built_bam(tmp_path):
    from test_gpu_hand_built_reads import CONTIGS, _soa, build_corpus
    c = build_corpus()
    refs = c.refs()
    fa = tmp_path / "ref.fa"
    with open(fa, "w") as fh:
        for name, n in CONTIGS:
            s = refs.fetch(name, 0, n)
            fh.write(">%s\n" % name + "".join(s[i:i + 60] + "\n" for i in range(0, n, 60)))
    bed = tmp_path / "t.bed"
    bed.write_text("".join("%s\t%d\t%d\n" % iv for iv in c.all_intervals()))
    path = str(tmp_path / "reads.bam")
    bam.write_bam(path, _soa(c.records()), dict(CONTIGS), index=True, block=1000)
    extra = dict(mtDepth=50, rpb=3.0, threshold=8, mtDrop=1, hpLen=8)
    assert _cli_files(tmp_path, path, fa, str(bed), "host", extra) == _cli_files(tmp_path, path, fa, str(bed), "gpu", extra)
