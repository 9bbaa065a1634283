"""BAM/BGZF decode -> ReadsSoA (smcounter_b200/bam.py): write a synthetic panel as a BAM, read it back, compare every
buffer; identity parsing follows smCounter.py:319-325 and the NM lookup :329-334."""
import gzip
import os
import struct

import numpy as np
import pytest

from smcounter_b200 import bam
from smcounter_b200.synth import SynthSpec, make_panel

FIELDS = ("ref_id", "pos", "flag", "mapq", "nm", "l_seq", "seq_off", "qual_off", "cigar_off", "n_cigar", "umi", "frag_id", "seq",
          "qual", "cigar")


def _panel(seed=2):
    spec = SynthSpec(umis_per_locus=15, rpb=2.5, snv_every=30, snv_vaf=0.2, indel_every=40, indel_vaf=0.2, softclip_frac=0.2)
    ivs = [("chr1", 400, 460), ("chr2", 150, 170)]
    s, refs, _ = make_panel(ivs, spec, seed=seed)
    return s, refs, ivs


def _decoders():
    out = [False]
    try:
        from smcounter_b200 import _bamio
        _bamio.load()
        out.append(True)
    except ImportError:
        pass
    return out


@pytest.mark.parametrize("native", _decoders())
def test_bam_roundtrip(tmp_path, native):
    s, refs, ivs = _panel()
    path = str(tmp_path / "t.bam")
    bam.write_bam(path, s, refs.lengths)
    back = bam.read_bam(path, native=native)
    assert back.chroms == s.chroms and back.n == s.n
    for f in FIELDS:
        assert np.array_equal(getattr(s, f), getattr(back, f)), f
    from smcounter_b200.soa import umi_string
    # every packed code decodes to a barcode that packs back to it; names are kept only where they are needed (dictionary codes)
    assert all((c >> 63) or bam.umi_code(umi_string(c, back.umi_names), {}) == c for c in set(back.umi.tolist()))
    # it is a valid gzip stream and ends with the BGZF EOF marker
    raw = open(path, "rb").read()
    assert raw.endswith(bam._BGZF_EOF)
    assert gzip.decompress(raw)[:4] == b"BAM\x01"


@pytest.mark.parametrize("native", _decoders())
def test_bam_interval_filter_and_tags(tmp_path, native):
    s, refs, ivs = _panel(seed=5)
    path = str(tmp_path / "t.bam")
    # NM stored as a 32-bit int after other tags of every encoding class
    extra = b"RGZgrp1\x00" + b"XAc\xff" + b"XBS\x01\x02" + b"XCf\x00\x00\x80\x3f" + b"XDBc\x03\x00\x00\x00\x01\x02\x03" + b"XEH1AE3\x00"
    bam.write_bam(path, s, refs.lengths, nm_type="i", extra_tags=extra,
                  qname_fn=lambda i, fid, bc: "INST:1:FC:%d:%s:%d" % (fid, bc, 7))
    target = [ivs[1]]
    back = bam.read_bam(path, intervals=target, native=native)
    ends = s.ref_end()
    keep = np.flatnonzero((s.ref_id == 1) & (s.pos < target[0][2]) & (ends > target[0][1]))
    assert back.n == len(keep) > 0
    for f in ("pos", "flag", "mapq", "nm", "l_seq", "n_cigar", "umi"):
        assert np.array_equal(getattr(s, f)[keep], getattr(back, f)), f
    # fragment ids: same partition as the original, numbered by first appearance
    pairs = set(zip(s.frag_id[keep].tolist(), back.frag_id.tolist()))
    assert len(pairs) == len(set(back.frag_id.tolist())) == len(set(s.frag_id[keep].tolist()))
    assert np.array_equal(np.unique(back.frag_id, return_index=True)[1], np.sort(np.unique(back.frag_id, return_index=True)[1]))
    first_seen = [back.frag_id[i] for i in sorted(np.unique(back.frag_id, return_index=True)[1])]
    assert first_seen == list(range(len(first_seen)))


@pytest.mark.parametrize("native", _decoders())
def test_unmapped_dropped_and_missing_nm(tmp_path, native):
    s, refs, ivs = _panel(seed=8)
    s.flag = s.flag.copy()
    s.flag[3] |= 0x4
    path = str(tmp_path / "t.bam")
    bam.write_bam(path, s, refs.lengths)
    # strip the NM tag of every record by rewriting the raw stream
    raw = bam.bgzf_decompress(open(path, "rb").read())
    _, refs_hdr, first = bam.parse_header(raw)
    out = [raw[:first]]
    p = first
    while p < len(raw):
        bs = struct.unpack_from("<i", raw, p)[0]
        body = raw[p + 4:p + 4 + bs]
        assert body[-4:-1] == b"NMC"
        body = body[:-4]
        out.append(struct.pack("<i", len(body)) + body)
        p += 4 + bs
    with open(path, "wb") as fh:
        fh.write(bam.bgzf_compress(b"".join(out)))
    back = bam.read_bam(path, native=native)
    assert back.n == s.n - 1 and not (back.flag & 0x4).any()
    assert (back.nm == 0).all()                                    # smCounter.py:329-334: NM defaults to 0


def test_bgzf_multi_block_roundtrip():
    rng = np.random.default_rng(0)
    data = rng.integers(0, 4, size=300000, dtype=np.uint8).tobytes()
    comp = bam.bgzf_compress(data, block=40000)
    assert bam.bgzf_decompress(comp) == data
    with pytest.raises(ValueError):
        bam.bgzf_decompress(b"\x1f\x8b\x08\x00" + b"\x00" * 30)


def test_native_decoder_trim_mode_matches_trim_to_targets(tmp_path):
    """smc_bam_set_trim: the C++ decoder's stored windows and payload are exactly ReadsSoA.trim_to_targets() of the untrimmed
    decode (both for overlapping / adjacent intervals and reads with soft clips and indels)."""
    import numpy as np
    from smcounter_b200 import bam
    from smcounter_b200.synth import SynthSpec, make_panel
    ivs = [("chr1", 1000, 1100), ("chr1", 1090, 1120), ("chr1", 1120, 1130), ("chr2", 300, 380), ("chr1", 5000, 5060)]
    soa, refs, _ = make_panel(ivs, SynthSpec(umis_per_locus=30, rpb=3.0, indel_every=30, indel_vaf=0.1, softclip_frac=0.3), seed=9)
    path = str(tmp_path / "t.bam")
    bam.write_bam(path, soa, refs.lengths)
    want = bam.read_bam(path, ivs, native=True).trim_to_targets(ivs)
    got = bam.read_bam(path, ivs, native=True, trim=True)
    assert got.packed and got.store_lo is not None and (got.store_len < got.l_seq).any()
    for f in ("ref_id", "pos", "flag", "l_seq", "n_cigar", "umi", "frag_id", "store_lo", "store_len", "seq_off", "qual_off", "cigar_off", "qual", "cigar"):
        assert np.array_equal(getattr(got, f), getattr(want, f)), f
    # seq: identical up to the unused low nibble after an odd-length window
    assert got.seq.shape == want.seq.shape
    last = (want.seq_off + (want.store_len.astype(np.int64) + 1) // 2 - 1)[want.store_len % 2 == 1]
    mask = np.ones(len(want.seq), dtype=bool); mask[last] = False
    assert np.array_equal(got.seq[mask], want.seq[mask]) and np.array_equal(got.seq[last] >> 4, want.seq[last] >> 4)
    py = bam.read_bam(path, ivs, native=False, trim=True)
    assert np.array_equal(py.store_lo, want.store_lo) and np.array_equal(py.qual, want.qual)


def test_native_decoder_parallel_passes_equal_single_thread(tmp_path):
    """A file big enough (> 8 MiB inflated) for the decoder's parallel passes -- speculative record-boundary search per byte
    range, hash-partitioned fragment numbering, range-wise prefix sums -- decoded with 1, 2, 3 and 7 threads: identical arrays,
    trimmed and untrimmed; a truncated copy is refused with the serial walk's message."""
    import numpy as np
    from smcounter_b200 import bam
    from smcounter_b200.synth import SynthSpec, make_panel
    ivs = [("chr1", 1000, 1150), ("chr2", 300, 420), ("chr1", 5000, 5100)]
    soa, refs, _ = make_panel(ivs, SynthSpec(umis_per_locus=1500, rpb=4.0, indel_every=60, indel_vaf=0.05, softclip_frac=0.2), seed=12)
    path = str(tmp_path / "big.bam")
    bam.write_bam(path, soa, refs.lengths)
    assert soa.n * 330 > (9 << 20)
    fields = ("ref_id", "pos", "flag", "mapq", "nm", "l_seq", "n_cigar", "umi", "frag_id", "seq_off", "qual_off", "cigar_off", "seq", "qual", "cigar")
    for trim in (False, True):
        one = bam.read_bam(path, ivs, native=True, threads=1, trim=trim)
        assert one.n > 0.7 * soa.n
        for th in (2, 3, 7):
            r = bam.read_bam(path, ivs, native=True, threads=th, trim=trim)
            for f in fields + (("store_lo", "store_len") if trim else ()):
                assert np.array_equal(getattr(r, f), getattr(one, f)), (trim, th, f)
    whole = bam.read_bam(path, None, native=True, threads=5)
    for f in fields:
        assert np.array_equal(getattr(whole, f), getattr(soa, f)), f
    # truncation inside the record stream: re-compress a cut copy of the inflated stream
    raw = bam.bgzf_decompress(open(path, "rb").read())
    cut = str(tmp_path / "cut.bam")
    with open(cut, "wb") as fh:
        fh.write(bam.bgzf_compress(raw[:len(raw) - 1000], 1))
    with pytest.raises(ValueError, match="truncated BAM record"):
        bam.read_bam(cut, ivs, native=True, threads=4)


@pytest.mark.parametrize("native", _decoders())
def test_bgzf_streams_as_other_writers_make_them(tmp_path, native):
    """BGZF as written by tools other than ours: blocks of irregular sizes that cut records (and even the 4-byte block_size
    field) in two, every deflate flavour (stored blocks, fixed Huffman, dynamic Huffman at levels 1 and 9), an extra gzip
    subfield before the BC one, an empty block in the middle of the file and the standard EOF marker at the end."""
    import zlib
    s, refs, ivs = _panel(seed=11)
    path = str(tmp_path / "a.bam")
    bam.write_bam(path, s, refs.lengths)
    want = bam.read_bam(path, native=native)
    raw = bam.bgzf_decompress(open(path, "rb").read())
    rng = np.random.default_rng(7)
    flavours = [(0, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_FIXED), (1, zlib.Z_DEFAULT_STRATEGY), (9, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_HUFFMAN_ONLY)]
    out, p, k = [], 0, 0

    def block(chunk, level, strategy, extra_subfield):
        co = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
        c = co.compress(chunk) + co.flush()
        extra = (b"XY\x03\x00abc" if extra_subfield else b"") + b"BC\x02\x00"
        xlen = len(extra) + 2
        bsize = 12 + xlen + len(c) + 8 - 1
        return (b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff" + struct.pack("<H", xlen) + extra + struct.pack("<H", bsize) + c +
                struct.pack("<II", zlib.crc32(chunk) & 0xffffffff, len(chunk)))
    while p < len(raw):
        n = int(rng.choice([1, 3, 37, 501, 4099, 30011]))
        chunk = raw[p:p + n]
        level, strategy = flavours[k % len(flavours)]
        out.append(block(chunk, level, strategy, k % 3 == 1))
        if k == 5:
            out.append(block(b"", 6, zlib.Z_DEFAULT_STRATEGY, False))          # an empty block inside the file
        p += n
        k += 1
    out.append(bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000"))   # the EOF marker of the SAM specification
    path2 = str(tmp_path / "b.bam")
    with open(path2, "wb") as fh:
        fh.write(b"".join(out))
    got = bam.read_bam(path2, native=native)
    assert got.n == want.n > 0
    for f in FIELDS:
        assert np.array_equal(getattr(got, f), getattr(want, f)), f
    got_t = bam.read_bam(path2, intervals=ivs, native=native, threads=3) if native else bam.read_bam(path2, intervals=ivs, native=native)
    want_t = bam.read_bam(path, intervals=ivs, native=native)
    for f in FIELDS:
        assert np.array_equal(getattr(got_t, f), getattr(want_t, f)), f


def _native_inflate(comp: bytes, out_len: int):
    import ctypes as C
    from smcounter_b200 import _bamio
    lib = _bamio.load()
    src = np.frombuffer(comp + b"\x00" * 64, dtype=np.uint8).copy()        # the routine may read up to 64 bytes past the stream
    dst = np.full(out_len + 64, 0xAB, dtype=np.uint8)                        # canary behind the output
    rc = lib.smc_bam_inflate_raw(src.ctypes.data, len(comp), dst.ctypes.data, out_len)
    assert (dst[out_len:] == 0xAB).all(), "wrote past the output"
    return rc, dst[:out_len].tobytes()


@pytest.mark.skipif(len(_decoders()) < 2, reason="libsmc_bamio.so not built")
def test_own_inflate_equals_zlib_on_every_kind_of_stream():
    """csrc/smc_inflate.h (what the BAM decoder inflates BGZF blocks with) against zlib: random bytes of several entropies,
    text, BAM-like records, long runs, empty input; compression levels 0-9, default / fixed-Huffman / Huffman-only / RLE /
    filtered strategies, streams of several deflate blocks (Z_FULL_FLUSH); sizes around every boundary of the copy loops."""
    import zlib
    rng = np.random.default_rng(12)
    def corpus():
        yield b""
        yield b"a"
        yield b"ab" * 7
        for n in (1, 2, 7, 8, 9, 15, 16, 17, 255, 256, 257, 258, 259, 4095, 65280):
            yield bytes(rng.integers(0, 256, size=n, dtype=np.uint8))                       # incompressible
            yield bytes(rng.integers(0, 4, size=n, dtype=np.uint8))                         # 2 bits of entropy
            yield (b"ACGT" * (n // 4 + 1))[:n]                                               # period 4
            yield b"\x00" * n                                                                # one long run (distance 1)
            yield bytes(np.repeat(rng.integers(0, 256, size=n // 9 + 1, dtype=np.uint8), 9)[:n])
        yield (b"the quick brown fox jumps over the lazy dog. " * 900)[:40000]
        s, refs, _ = _panel(seed=3)
        p = "/tmp/_smc_inflate_case.bam"
        bam.write_bam(p, s, refs.lengths)
        yield bam.bgzf_decompress(open(p, "rb").read())[:65280]
        os.remove(p)
        yield bytes(rng.integers(0, 256, size=20000, dtype=np.uint8)) + b"\x07" * 20000 + bytes(rng.integers(0, 16, size=20000, dtype=np.uint8))
    n_streams = 0
    for data in corpus():
        for level in (0, 1, 4, 6, 9):
            for strategy in (zlib.Z_DEFAULT_STRATEGY, zlib.Z_FIXED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FILTERED):
                co = zlib.compressobj(level, zlib.DEFLATED, -15, 9, strategy)
                comp = co.compress(data) + co.flush()
                rc, got = _native_inflate(comp, len(data))
                assert rc == 0 and got == data, (len(data), level, strategy)
                n_streams += 1
        # several deflate blocks in one stream, of different kinds
        co = zlib.compressobj(6, zlib.DEFLATED, -15)
        half = len(data) // 2
        comp = co.compress(data[:half]) + co.flush(zlib.Z_FULL_FLUSH) + co.compress(data[half:]) + co.flush()
        rc, got = _native_inflate(comp, len(data))
        assert rc == 0 and got == data
    assert n_streams > 1500


@pytest.mark.skipif(len(_decoders()) < 2, reason="libsmc_bamio.so not built")
def test_own_inflate_rejects_what_it_cannot_prove_right():
    """Wrong output size, truncated input, flipped bits: the routine must never write outside the output it was given (canary
    checked in _native_inflate) and must return an error or -- for a flipped bit that still decodes -- output of the stated size;
    it never crashes.  (The BAM decoder hands rejected blocks to zlib.)"""
    import zlib
    rng = np.random.default_rng(5)
    data = bytes(rng.integers(0, 8, size=30000, dtype=np.uint8)) + b"GATTACA" * 500
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    comp = co.compress(data) + co.flush()
    assert _native_inflate(comp, len(data))[0] == 0
    assert _native_inflate(comp, len(data) - 1)[0] == -1
    assert _native_inflate(comp, len(data) + 1)[0] == -1
    for cut in (1, 2, 10, len(comp) // 2, len(comp) - 1):
        assert _native_inflate(comp[:cut], len(data))[0] == -1
    bad = 0
    for k in range(400):
        b = bytearray(comp)
        pos = int(rng.integers(0, len(b)))
        b[pos] ^= 1 << int(rng.integers(0, 8))
        rc, got = _native_inflate(bytes(b), len(data))
        assert rc in (0, -1)
        bad += rc == -1 or got != data
    assert bad > 300                     # nearly every flip is caught by the stream's own consistency (size, codes, distances)
    for k in range(200):                 # garbage
        junk = bytes(rng.integers(0, 256, size=int(rng.integers(1, 400)), dtype=np.uint8))
        assert _native_inflate(junk, 1000)[0] in (0, -1)


def test_own_inflate_under_address_sanitizer(tmp_path):
    """csrc/smc_inflate.h compiled with -fsanitize=address,undefined (tests/inflate_asan_harness.cpp) over ~4 600 streams:
    every zlib flavour of eight data sets, each with bit flips, truncations, overwritten bytes and wrong stated sizes, plus
    3 000 random byte strings -- input buffers carry exactly the documented 64 bytes of slack, output buffers none.  No
    sanitizer report, every valid stream decoded to zlib's bytes."""
    import shutil
    import subprocess
    import zlib
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    here = os.path.dirname(os.path.abspath(__file__))
    exe = str(tmp_path / "h")
    r = subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-fsanitize=address,undefined", "-fno-omit-frame-pointer",
                        "-I", os.path.join(here, "..", "smcounter_b200", "csrc"), "-o", exe, os.path.join(here, "inflate_asan_harness.cpp")],
                       capture_output=True, text=True)
    if r.returncode != 0:
        pytest.skip("sanitizer runtime not available: " + r.stderr[-200:])
    rng = np.random.default_rng(99)
    n = 0
    with open(tmp_path / "cases.bin", "wb") as out:
        def put(comp, outlen, ok, data=b""):
            out.write(struct.pack("<IIB", len(comp), outlen, ok) + comp + (data if ok else b""))
        datas = [b"", b"x", bytes(rng.integers(0, 256, size=3000, dtype=np.uint8)), bytes(rng.integers(0, 4, size=50000, dtype=np.uint8)), b"ACGT" * 9000,
                 b"\0" * 65280, (b"hello world, hello deflate. " * 3000)[:65000], bytes(np.repeat(rng.integers(0, 256, size=7000, dtype=np.uint8), 9))[:60000]]
        for d in datas:
            for lvl in (0, 1, 6, 9):
                for st in (zlib.Z_DEFAULT_STRATEGY, zlib.Z_FIXED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE):
                    co = zlib.compressobj(lvl, zlib.DEFLATED, -15, 9, st)
                    c = co.compress(d) + co.flush()
                    put(c, len(d), 1, d); n += 1
                    for k in range(12):
                        b = bytearray(c)
                        if not b:
                            continue
                        mode = k % 4
                        if mode == 0:
                            b[int(rng.integers(0, len(b)))] ^= 1 << int(rng.integers(0, 8))
                        elif mode == 1:
                            b = b[:int(rng.integers(0, len(b)))]
                        elif mode == 2:
                            pos = int(rng.integers(0, len(b)))
                            b[pos:pos + 4] = bytes(rng.integers(0, 256, size=min(4, len(b) - pos), dtype=np.uint8))
                        put(bytes(b), len(d) if mode != 3 else max(0, len(d) + int(rng.integers(-3, 4))), 0); n += 1
        for k in range(3000):
            put(bytes(rng.integers(0, 256, size=int(rng.integers(0, 600)), dtype=np.uint8)), int(rng.integers(0, 5000)), 0); n += 1
    r = subprocess.run([exe, str(tmp_path / "cases.bin")], capture_output=True, text=True)
    assert r.returncode == 0 and "runtime error" not in r.stderr and "AddressSanitizer" not in r.stderr, r.stdout[-500:] + r.stderr[-2000:]
    assert ("%d cases" % n) in r.stdout and " 0 wrong" in r.stdout


@pytest.mark.skipif(len(_decoders()) < 2, reason="libsmc_bamio.so not built")
def test_native_decoder_counts_the_stored_qualities(tmp_path):
    """smc_bam_reads.qual_hist (counted during the copy pass) == a histogram of the decoded qual[] -- with and without trimming,
    any thread count -- and the upload codebook built from it equals the one from smc_soa_qual_hist."""
    from smcounter_b200 import _bamio
    s, refs, ivs = _panel(seed=21)
    path = str(tmp_path / "q.bam")
    bam.write_bam(path, s, refs.lengths)
    for trim in (False, True):
        for threads in (1, 4):
            r = bam.read_bam(path, intervals=ivs, native=True, threads=threads, trim=trim)
            h = r.__dict__["_qual_hist"]
            assert np.array_equal(h, np.bincount(r.qual, minlength=256).astype(np.uint64))
            cb = dict(_bamio.upload_codebook(r))
            r.__dict__.pop("_qual_hist"); r.__dict__.pop("_upload_codebook")
            cb2 = _bamio.upload_codebook(r)
            assert cb["qual_bits"] == cb2["qual_bits"] and np.array_equal(cb["qual_lut"], cb2["qual_lut"]) and np.array_equal(cb["code_of"], cb2["code_of"])


_OOM_CHILD = r"""
import resource, sys
from smcounter_b200 import _bamio, bam
lib = _bamio.load()
decode = lib.smc_bam_decode

def limited(*args):
    # from here on the process may map 1 MiB more than it has (VmData); the file is already inflated
    with open("/proc/self/status") as fh:
        vm_data = next(int(l.split()[1]) for l in fh if l.startswith("VmData:")) << 10
    resource.setrlimit(resource.RLIMIT_DATA, (vm_data + (1 << 20), resource.getrlimit(resource.RLIMIT_DATA)[1]))
    try:
        bytearray(8 << 20)
        print("limit not enforced")
        sys.exit(0)
    except MemoryError:
        pass
    return decode(*args)

lib.smc_bam_decode = limited
try:
    bam.read_bam(sys.argv[1], [("chr1", 0, 1 << 20), ("chr2", 0, 1 << 20)], native=True, threads=1, trim=True)
    print("decoded")
except ValueError as e:
    print("ValueError:", e)
"""


@pytest.mark.skipif(len(_decoders()) < 2, reason="libsmc_bamio.so not built")
def test_native_decoder_out_of_memory_is_an_error(tmp_path):
    """A decode whose tables and output arrays do not fit in memory (a child process, one thread, its data limit set just above
    what it uses before smc_bam_decode runs) raises ValueError('out of memory for ...'): the decoder checks its allocations
    instead of writing through a null pointer."""
    import subprocess
    import sys
    s, refs, _ = make_panel([("chr1", 1000, 1150), ("chr2", 300, 420)], SynthSpec(umis_per_locus=3000, rpb=4.0), seed=4)
    path = str(tmp_path / "oom.bam")
    bam.write_bam(path, s, refs.lengths)
    assert s.n * 56 > (2 << 20)                              # record offsets and the record table alone need more than 2 MiB
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", _OOM_CHILD, path], cwd=root, capture_output=True, text=True)
    if "limit not enforced" in r.stdout:
        pytest.skip("RLIMIT_DATA is not enforced here")
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.startswith("ValueError: out of memory for "), r.stdout + r.stderr[-2000:]


def _random_code_lengths(rng, n_symbols_used, alphabet, must_have=(), deep=False):
    """Lengths (<= 15) of a COMPLETE prefix code over ``n_symbols_used`` random symbols of ``alphabet`` (others 0)."""
    leaves = [0]
    while len(leaves) < n_symbols_used:
        cand = [i for i, d in enumerate(leaves) if d < 15]
        i = (max(cand, key=lambda k: leaves[k]) if deep and rng.random() < 0.8 else int(rng.choice(cand)))
        d = leaves.pop(i)
        leaves += [d + 1, d + 1]
    syms = list(must_have) + [int(x) for x in rng.permutation([s for s in range(alphabet) if s not in must_have])][:n_symbols_used - len(must_have)]
    lens = [0] * alphabet
    for s, d in zip(rng.permutation(syms), leaves):
        lens[int(s)] = max(d, 1)
    return lens


def _canonical_codes(lens):
    count = [0] * 16
    for l in lens:
        count[l] += 1
    count[0] = 0
    code, nxt = 0, [0] * 16
    for l in range(1, 16):
        code = (code + count[l - 1]) << 1
        nxt[l] = code
    out = {}
    for s, l in enumerate(lens):
        if l:
            out[s] = (nxt[l], l)
            nxt[l] += 1
    return out


class _BitWriter:
    def __init__(self):
        self.acc, self.n, self.out = 0, 0, bytearray()

    def bits(self, value, nbits):                 # LSB first
        self.acc |= value << self.n
        self.n += nbits
        while self.n >= 8:
            self.out.append(self.acc & 255)
            self.acc >>= 8
            self.n -= 8

    def code(self, cl):                           # Huffman codes go in MSB first
        c, l = cl
        self.bits(int(format(c, "0%db" % l)[::-1], 2), l)

    def done(self):
        if self.n:
            self.out.append(self.acc & 255)
        return bytes(self.out)


@pytest.mark.skipif(len(_decoders()) < 2, reason="libsmc_bamio.so not built")
def test_own_inflate_on_hand_made_dynamic_blocks():
    """Dynamic-Huffman blocks written bit by bit with RANDOM complete codes -- code lengths up to 15 on both alphabets (the
    secondary tables of the decoder), single-code distance alphabets, every length / distance symbol with its extra bits --
    decoded by zlib (which validates the encoder) and by csrc/smc_inflate.h."""
    import zlib
    LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
    LEN_EXTRA = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
    DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577]
    DIST_EXTRA = [0, 0, 0, 0] + [k for k in range(1, 14) for _ in (0, 1)]
    ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
    rng = np.random.default_rng(31)
    deepest = 0
    for case in range(120):
        deep = case % 2 == 0
        n_lit = int(rng.integers(2, 286))
        lit_lens = _random_code_lengths(rng, n_lit, 286, must_have=(256,), deep=deep)
        n_dist = int(rng.integers(1, 31))
        dist_lens = _random_code_lengths(rng, n_dist, 30, deep=deep) if n_dist > 1 else [0] * 30
        if n_dist == 1:
            dist_lens[int(rng.integers(0, 30))] = 1                      # one distance code: the incomplete code RFC 1951 allows
        deepest = max(deepest, max(lit_lens), max(dist_lens))
        lit_codes, dist_codes = _canonical_codes(lit_lens), _canonical_codes(dist_lens)
        pre_lens = [0] * 19
        for k, s in enumerate(rng.permutation(19)):
            pre_lens[int(s)] = 4 if k < 13 else 5                        # 13/16 + 6/32 = 1: complete
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
        rc, got = _native_inflate(stream, len(out))
        assert rc == 0 and got == bytes(out), case
    assert deepest == 15


@pytest.mark.skipif(len(_decoders()) < 2, reason="libsmc_bamio.so not built")
def test_dictionary_coded_barcodes_native_equals_python(tmp_path):
    """Barcodes that do not pack into 64 bits (an 'N', more than 31 nt) get dictionary codes in order of first appearance: the
    C++ decoder (whose dictionary pass runs only when such a barcode exists) and the Python walker must agree, and a file
    without any such barcode must come out without a dictionary."""
    from smcounter_b200.soa import umi_string
    s, refs, ivs = _panel(seed=17)
    odd = {3: "ACGTNACGTACG", 11: "A" * 40, 12: "ACGTNACGTACG", 30: "TTTTGGGGNNNN"}

    def qname(i, fid, bc):
        return "M1:F%d:%s:%d" % (fid, odd.get(i % 40, bc), 1)
    for fn, expect_dict in ((qname, True), (None, False)):
        path = str(tmp_path / ("d%d.bam" % expect_dict))
        bam.write_bam(path, s, refs.lengths, qname_fn=fn)
        a = bam.read_bam(path, native=True, threads=3)
        b = bam.read_bam(path, native=False)
        assert a.n == b.n
        for f in FIELDS:
            assert np.array_equal(getattr(a, f), getattr(b, f)), f
        da, db = ({k: v for k, v in x.umi_names.items() if k >> 63} for x in (a, b))      # the Python walker also names the packed codes
        assert da == db and bool(da) == expect_dict
        if expect_dict:
            assert {umi_string(int(c), a.umi_names) for c in a.umi.tolist() if c >> 63} == {"ACGTNACGTACG", "A" * 40, "TTTTGGGGNNNN"}
