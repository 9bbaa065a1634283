"""The planning entries of libsmc_bamio (smc_bam_open_header, smc_bam_plan, smc_bam_read_blocks): the listed blocks, inflated with
zlib and placed at their stream offsets, are exactly the stream the host decode walks -- whole file and through the .bai, for
several BGZF block sizes -- and index errors carry the host decode's messages."""
import zlib

import pytest

from smcounter_b200 import bam
from smcounter_b200.synth import SynthSpec, make_panel

_bamio = pytest.importorskip("smcounter_b200._bamio")


def _stream(buf, blocks, raw_bytes):
    out = bytearray(raw_bytes)
    for (coff, clen, uoff, isize, lo, hi) in blocks:
        u = zlib.decompress(bytes(buf[coff:coff + clen]), -15) if isize else b""
        assert len(u) == isize
        out[uoff:uoff + hi - lo] = u[lo:hi]
    return bytes(out)


@pytest.mark.parametrize("block", [512, 3000, 0xff00])
def test_planned_blocks_reproduce_the_decoded_stream(tmp_path, block):
    _bamio.load()
    ivs = [("chr1", 400, 460), ("chr2", 150, 170), ("chr1", 2000, 2040)]
    s, refs, _ = make_panel(ivs, SynthSpec(umis_per_locus=20, rpb=2.5, softclip_frac=0.2), seed=3)
    path = str(tmp_path / "t.bam")
    bam.write_bam(path, s, refs.lengths, index=True, block=block)
    raw = bam.bgzf_decompress(open(path, "rb").read())
    buf, blocks, raw_bytes, first = _bamio.plan_blocks(path)
    assert (buf[-64:] == 0).all()
    assert _stream(buf, blocks, raw_bytes) == raw and first == bam.parse_header(raw)[2]
    names = list(s.chroms)
    for sub in (ivs, ivs[1:2], [("chr1", 10 ** 6, 10 ** 6 + 10)]):
        buf, blocks, raw_bytes, first = _bamio.plan_blocks(path, sub, index=path + ".bai")
        chunks = bam.bai_chunks(bam.read_bai(path + ".bai", len(names)), names, sub)
        assert _stream(buf, blocks, raw_bytes) == bam.read_chunks(path, chunks, path + ".bai") and first == 0
    # intervals without an index: the whole file
    buf, blocks, raw_bytes, first = _bamio.plan_blocks(path, ivs)
    assert _stream(buf, blocks, raw_bytes) == raw


def test_bad_chunk_gives_the_host_decode_error(tmp_path):
    ivs = [("chr1", 400, 460)]
    s, refs, _ = make_panel(ivs, SynthSpec(umis_per_locus=10, rpb=2.0), seed=4)
    path = str(tmp_path / "t.bam")
    bam.write_bam(path, s, refs.lengths, index=True, block=2000)
    bai = bytearray(open(path + ".bai", "rb").read())
    # every chunk of the index points past the end of the file
    import struct
    size = len(open(path, "rb").read())
    p = 8
    n_bin = struct.unpack_from("<i", bai, p)[0]; p += 4
    for _ in range(n_bin):
        b, n_chunk = struct.unpack_from("<Ii", bai, p); p += 8
        for c in range(n_chunk):
            if b != 37450:
                struct.pack_into("<QQ", bai, p + 16 * c, (size + 100) << 16, (size + 200) << 16)
        p += 16 * n_chunk
    open(path + ".bai", "wb").write(bytes(bai))
    with pytest.raises(IOError) as host:
        bam.read_bam(path, ivs, native=True)
    with pytest.raises(IOError) as plan:
        _bamio.plan_blocks(path, ivs, index=path + ".bai")
    assert str(plan.value) == str(host.value) and "points past the end" in str(plan.value)
