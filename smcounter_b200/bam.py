"""BAM (BGZF) <-> ReadsSoA, the caller side of the hot path (SURVEY.md section 8f.1).

The reference reads its input through pysam (``pysam.AlignmentFile(bamFile, 'rb')`` + ``pileup``,
smCounter.py:275,316) and re-decodes every read once per covered locus.  Here every BAM record is decoded ONCE
into the flat structure-of-arrays buffers that cross the C-ABI (include/smc_b200.h: smc_reads_soa).  pysam /
htslib are third-party and not installed in this image, so the container format is restated from the SAM/BAM
specification (SAMv1 section 4): BGZF = concatenated gzip members whose extra field 'BC' holds the block size;
BAM = magic, text header, reference list, then records
``block_size refID pos l_read_name mapq bin n_cigar_op flag l_seq next_refID next_pos tlen read_name cigar seq qual tags``.

Per-record identity follows smCounter.py:319-325 (``readid = ':'.join(parts[:-2])``, ``BC = parts[-2]``) and the
NM lookup smCounter.py:329-334 (first NM tag, 0 when absent).  Unmapped records are dropped (htslib never piles them
up); no other flag filtering is applied (the reference uses ``stepper='nofilter'``).

``read_bam`` uses the native decoder (csrc/smc_bamio.cpp -> libsmc_bamio.so) when it is built and falls back to the
pure-Python record walker otherwise; both produce identical buffers (tests/test_bam_io.py).  With target intervals and
a current .bai beside the BAM (SAMv1 section 5.2), both read and inflate only the index chunks the targets need, and give
the same buffers as a whole-file decode (tests/test_bam_index.py).  This is host-side input decoding, not the calling hot
path: the hot path itself has no CPU implementation.
"""
from __future__ import annotations

import os
import struct
import zlib

import numpy as np

from .soa import ReadsSoA, umi_code

_BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


# ------------------------------------------------------------------------------------------------------------------
# BGZF
# ------------------------------------------------------------------------------------------------------------------
def _bgzf_blocks(data: bytes):
    """(offset, inflated bytes) of every BGZF block of ``data``, in order."""
    off = 0
    n = len(data)
    while off < n:
        if data[off:off + 4] != b"\x1f\x8b\x08\x04":
            raise ValueError("not a BGZF block at offset %d" % off)
        xlen = struct.unpack_from("<H", data, off + 10)[0]
        p = off + 12
        bsize = None
        end = p + xlen
        while p < end:
            si1, si2, slen = data[p], data[p + 1], struct.unpack_from("<H", data, p + 2)[0]
            if si1 == 66 and si2 == 67 and slen == 2:
                bsize = struct.unpack_from("<H", data, p + 4)[0]
            p += 4 + slen
        if bsize is None:
            raise ValueError("BGZF block without BC subfield at offset %d" % off)
        if off + bsize + 1 > n:
            raise ValueError("truncated BGZF block at offset %d" % off)
        cdata = data[off + 12 + xlen: off + bsize + 1 - 8]
        isize = struct.unpack_from("<I", data, off + bsize + 1 - 4)[0]
        yield off, (zlib.decompress(cdata, -15) if isize else b"")
        off += bsize + 1


def bgzf_decompress(data: bytes) -> bytes:
    """Inflate every BGZF block of ``data`` and concatenate."""
    return b"".join(u for _, u in _bgzf_blocks(data))


def _bgzf_block_list(raw: bytes, level: int = 6, block: int = 0xff00):
    """The BGZF blocks of ``raw`` (``block`` inflated bytes each, the last one shorter), without the EOF marker."""
    out = []
    for i in range(0, len(raw), block):
        chunk = raw[i:i + block]
        co = zlib.compressobj(level, zlib.DEFLATED, -15)
        c = co.compress(chunk) + co.flush()
        bsize = 12 + 6 + len(c) + 8 - 1
        out.append(b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", bsize) + c +
                   struct.pack("<II", zlib.crc32(chunk) & 0xffffffff, len(chunk)))
    return out


def bgzf_compress(raw: bytes, level: int = 6, block: int = 0xff00) -> bytes:
    return b"".join(_bgzf_block_list(raw, level, block) + [_BGZF_EOF])


# ------------------------------------------------------------------------------------------------------------------
# BAM header
# ------------------------------------------------------------------------------------------------------------------
def parse_header(raw: bytes):
    """Returns (text, [(name, length)], offset of the first record)."""
    if raw[:4] != b"BAM\x01":
        raise ValueError("not a BAM file (bad magic)")
    l_text = struct.unpack_from("<i", raw, 4)[0]
    text = raw[8:8 + l_text].decode("ascii", "replace")
    p = 8 + l_text
    n_ref = struct.unpack_from("<i", raw, p)[0]
    p += 4
    refs = []
    for _ in range(n_ref):
        l_name = struct.unpack_from("<i", raw, p)[0]
        name = raw[p + 4:p + 4 + l_name - 1].decode()
        l_ref = struct.unpack_from("<i", raw, p + 4 + l_name)[0]
        refs.append((name, l_ref))
        p += 8 + l_name
    return text, refs, p


_TAG_SIZE = {ord("A"): 1, ord("c"): 1, ord("C"): 1, ord("s"): 2, ord("S"): 2, ord("i"): 4, ord("I"): 4, ord("f"): 4}
_TAG_FMT = {ord("c"): "<b", ord("C"): "<B", ord("s"): "<h", ord("S"): "<H", ord("i"): "<i", ord("I"): "<I"}


def _first_nm(raw, p, end):
    """Value of the first NM tag in raw[p:end], or 0 (smCounter.py:329-334)."""
    while p + 3 <= end:
        t0, t1, ty = raw[p], raw[p + 1], raw[p + 2]
        p += 3
        if ty in _TAG_SIZE:
            if t0 == 78 and t1 == 77 and ty in _TAG_FMT:
                return int(struct.unpack_from(_TAG_FMT[ty], raw, p)[0])
            p += _TAG_SIZE[ty]
        elif ty in (90, 72):                       # Z, H
            q = raw.index(b"\x00", p)
            p = q + 1
        elif ty == 66:                             # B
            sub = raw[p]
            cnt = struct.unpack_from("<i", raw, p + 1)[0]
            p += 5 + cnt * _TAG_SIZE.get(sub, 1)
        else:
            break
    return 0


def _intervals_by_ref(intervals, ref_names):
    """ref index -> (sorted starts, running max of ends) for the 'does this read touch a target' test."""
    by = {}
    idx = {n: i for i, n in enumerate(ref_names)}
    for (c, s, e) in intervals or ():
        if c in idx and e > s:
            by.setdefault(idx[c], []).append((s, e))
    out = {}
    for r, v in by.items():
        v.sort()
        starts = np.asarray([s for s, _ in v], dtype=np.int64)
        ends = np.maximum.accumulate(np.asarray([e for _, e in v], dtype=np.int64))
        out[r] = (starts, ends)
    return out


def _touches(tab, rid, s, e):
    t = tab.get(rid)
    if t is None:
        return False
    starts, maxend = t
    k = int(np.searchsorted(starts, e, side="left"))     # intervals starting before the read end
    return k > 0 and int(maxend[k - 1]) > s


def decode_records_py(raw: bytes, first: int, ref_names, intervals=None) -> ReadsSoA:
    """Pure-Python record walker (reference implementation of the decoder; the native one must agree with it)."""
    tab = _intervals_by_ref(intervals, ref_names) if intervals is not None else None
    cols = {k: [] for k in ("ref_id", "pos", "flag", "mapq", "nm", "l_seq", "n_cigar", "umi", "frag")}
    seqs, quals, cigs = [], [], []
    umitab, fragtab, names = {}, {}, {}
    p = first
    n = len(raw)
    unpack = struct.Struct("<iiBBHHHiiii").unpack_from
    while p + 4 <= n:
        bs = struct.unpack_from("<i", raw, p)[0]
        rec_end = p + 4 + bs
        refID, pos, l_rn, mapq, _bin, n_cig, flag, l_seq, _nr, _np, _tl = unpack(raw, p + 4)
        q = p + 36
        qname = raw[q:q + l_rn - 1].decode()
        q += l_rn
        cig = np.frombuffer(raw, dtype="<u4", count=n_cig, offset=q)
        q += 4 * n_cig
        sb = (l_seq + 1) // 2
        p = rec_end
        if flag & 0x4 or refID < 0:
            continue
        if tab is not None:
            ops = cig & 15
            reflen = int(((cig >> 4)[(ops == 0) | (ops == 2) | (ops == 3) | (ops == 7) | (ops == 8)]).sum())
            if not _touches(tab, refID, pos, pos + reflen):
                continue
        parts = qname.split(":")
        bc = parts[-2] if len(parts) >= 2 else ""
        readid = ":".join(parts[:-2])
        code = umi_code(bc, umitab)
        names[code] = bc
        fk = (bc, readid)
        fid = fragtab.get(fk)
        if fid is None:
            fid = fragtab[fk] = len(fragtab)
        cols["ref_id"].append(refID); cols["pos"].append(pos); cols["flag"].append(flag); cols["mapq"].append(mapq)
        cols["nm"].append(_first_nm(raw, q + sb + l_seq, rec_end)); cols["l_seq"].append(l_seq); cols["n_cigar"].append(n_cig)
        cols["umi"].append(code); cols["frag"].append(fid)
        cigs.append(cig)
        seqs.append(np.frombuffer(raw, dtype=np.uint8, count=sb, offset=q))
        quals.append(np.frombuffer(raw, dtype=np.uint8, count=l_seq, offset=q + sb))
    return _assemble(cols, seqs, quals, cigs, list(ref_names), names)


def _assemble(cols, seqs, quals, cigs, chroms, names):
    l_seq = np.asarray(cols["l_seq"], dtype=np.int32)
    n_cigar = np.asarray(cols["n_cigar"], dtype=np.uint16)
    ex = lambda lens: np.concatenate(([0], np.cumsum(lens, dtype=np.int64)))[:-1].astype(np.int64)
    cat = lambda xs, dt: np.concatenate(xs).astype(dt, copy=False) if xs else np.zeros(0, dt)
    return ReadsSoA(
        ref_id=np.asarray(cols["ref_id"], dtype=np.int32), pos=np.asarray(cols["pos"], dtype=np.int32),
        flag=np.asarray(cols["flag"], dtype=np.uint16), mapq=np.asarray(cols["mapq"], dtype=np.uint8),
        nm=np.asarray(cols["nm"], dtype=np.int32), l_seq=l_seq, seq_off=ex((l_seq.astype(np.int64) + 1) // 2),
        qual_off=ex(l_seq.astype(np.int64)), cigar_off=ex(n_cigar.astype(np.int64)), n_cigar=n_cigar,
        umi=np.asarray(cols["umi"], dtype=np.uint64), frag_id=np.asarray(cols["frag"], dtype=np.uint32),
        seq=cat(seqs, np.uint8), qual=cat(quals, np.uint8), cigar=cat(cigs, np.uint32), chroms=chroms, umi_names=names)


# ------------------------------------------------------------------------------------------------------------------
# BAM index (.bai, SAMv1 section 5.2): region access without inflating the whole file
# ------------------------------------------------------------------------------------------------------------------
_PSEUDO_BIN = 37450          # per-reference metadata: (first, last) virtual offsets and (mapped, unmapped) counts


def find_index(path: str):
    """The .bai that ``read_bam`` uses for ``path``: ``<path>.bai`` or ``<path without .bam>.bai`` (samtools' two names).
    None when there is none, or when it is older than the BAM -- a stale index can miss reads, so that gets a warning line and
    the whole file is decoded."""
    cands = [path + ".bai"] + ([path[:-4] + ".bai"] if path.endswith(".bam") else [])
    for idx in cands:
        if os.path.exists(idx):
            if os.path.getmtime(idx) < os.path.getmtime(path):
                print("warning: BAM index %s is older than %s; decoding the whole file instead" % (idx, path))
                return None
            return idx
    return None


def read_bai(index_path: str, n_ref: int):
    """[(bins {bin: [(beg, end)]}, linear [offset])] per reference; the pseudo-bin is skipped.  IOError naming the index
    when it is malformed or its reference count is not ``n_ref``."""
    with open(index_path, "rb") as fh:
        d = fh.read()
    try:
        if d[:4] != b"BAI\x01":
            raise IOError("BAM index %s: bad magic (not a .bai file)" % index_path)
        got = struct.unpack_from("<i", d, 4)[0]
        if got != n_ref:
            raise IOError("BAM index %s: n_ref is %d but the BAM header has %d references" % (index_path, got, n_ref))
        p, refs = 8, []
        for _ in range(n_ref):
            n_bin = struct.unpack_from("<i", d, p)[0]
            p += 4
            bins = {}
            for _ in range(n_bin):
                b, n_chunk = struct.unpack_from("<Ii", d, p)
                p += 8
                ch = struct.unpack_from("<%dQ" % (2 * n_chunk), d, p)
                p += 16 * n_chunk
                if b != _PSEUDO_BIN:
                    bins.setdefault(b, []).extend(zip(ch[0::2], ch[1::2]))
            n_intv = struct.unpack_from("<i", d, p)[0]
            p += 4
            refs.append((bins, list(struct.unpack_from("<%dQ" % n_intv, d, p))))
            p += 8 * n_intv
    except struct.error:
        raise IOError("BAM index %s: truncated or malformed" % index_path) from None
    if len(d) not in (p, p + 8):                            # nothing, or the optional n_no_coor
        raise IOError("BAM index %s: truncated or malformed" % index_path)
    return refs


def _reg2bins(beg, end):
    """SAMv1 section 5.3: the bins that may hold a record overlapping [beg, end)."""
    end -= 1
    out = [0]
    for first, shift in ((1, 26), (9, 23), (73, 20), (585, 17), (4681, 14)):
        out.extend(range(first + (beg >> shift), first + (end >> shift) + 1))
    return out


def bai_chunks(bai, ref_names, intervals):
    """The chunks [(beg, end)] (virtual offsets) that hold every record touching ``intervals``: the bins of each interval,
    less the chunks that end before its first 16 kbp window's linear-index offset; sorted, and merged where they overlap or
    share a BGZF block (which adds only whole records in between, and inflates every block once)."""
    idx = {n: i for i, n in enumerate(ref_names)}
    ch = []
    for (c, s, e) in intervals:
        r = idx.get(c)
        beg, end = max(0, s), min(e, 1 << 29)
        if r is None or r >= len(bai) or end <= beg:
            continue
        bins, lin = bai[r]
        min_off = lin[min(beg >> 14, len(lin) - 1)] if lin else 0
        for b in _reg2bins(beg, end):
            ch.extend(x for x in bins.get(b, ()) if x[1] > min_off and x[1] > x[0])
    merged = []
    for beg, end in sorted(ch):
        if merged and (beg >> 16) <= (merged[-1][1] >> 16):
            merged[-1][1] = max(merged[-1][1], end)
        else:
            merged.append([beg, end])
    return [tuple(m) for m in merged]


def _block_len(fh, off):
    fh.seek(off)
    head = fh.read(12)
    if len(head) < 12 or head[:2] != b"\x1f\x8b":
        return None
    xlen = struct.unpack_from("<H", head, 10)[0]
    extra = fh.read(xlen)
    p = 0
    while p + 6 <= len(extra):
        slen = struct.unpack_from("<H", extra, p + 2)[0]
        if extra[p:p + 2] == b"BC" and slen == 2:
            return struct.unpack_from("<H", extra, p + 4)[0] + 1
        p += 4 + slen
    return None


def read_header_blocks(fh):
    """(text, [(name, length)]) from the BGZF blocks at the start of ``fh``, inflated one at a time until the reference list
    is complete."""
    raw, off = b"", 0
    while True:
        n = _block_len(fh, off)
        if n is None:
            raise ValueError("not a BGZF block at offset %d" % off)
        fh.seek(off)
        raw += bgzf_decompress(fh.read(n))
        off += n
        if len(raw) < 4:
            continue
        try:
            text, refs, _first = parse_header(raw)
            return text, refs
        except (struct.error, IndexError, UnicodeDecodeError):
            continue


def read_chunks(path: str, chunks, index_path: str) -> bytes:
    """The inflated bytes of ``chunks`` (merged, sorted), concatenated: a record chain.  Only their compressed byte ranges are
    read.  IOError naming the index when a chunk points past the end of the file or not at BGZF blocks."""
    size = os.path.getsize(path)
    out = []
    with open(path, "rb") as fh:
        for beg, end in chunks:
            cbeg, ubeg, cend, uend = beg >> 16, beg & 0xFFFF, end >> 16, end & 0xFFFF
            stop = cend
            if cbeg >= size or cend > size or (cend == size and uend):
                raise IOError("BAM index %s: chunk [%d, %d) points past the end of %s" % (index_path, beg, end, path))
            if uend:
                n = _block_len(fh, cend) if cend < size else None
                if n is None:
                    raise IOError("BAM index %s: chunk end at virtual offset %d is not in a BGZF block of %s" % (index_path, end, path))
                stop = cend + n
            if stop > size or cbeg >= size:
                raise IOError("BAM index %s: chunk [%d, %d) points past the end of %s" % (index_path, beg, end, path))
            fh.seek(cbeg)
            try:
                blocks = list(_bgzf_blocks(fh.read(stop - cbeg)))
            except (ValueError, zlib.error, struct.error) as e:
                raise IOError("BAM index %s: chunk [%d, %d) does not point at BGZF blocks of %s (%s)" % (index_path, beg, end, path, e)) from None
            if uend and blocks[-1][0] != cend - cbeg:
                raise IOError("BAM index %s: chunk [%d, %d) does not point at BGZF blocks of %s" % (index_path, beg, end, path))
            data = [u for _, u in blocks]
            if uend:
                data[-1] = data[-1][:uend]
            data[0] = data[0][ubeg:]
            out.extend(data)
    return b"".join(out)


def read_bam(path: str, intervals=None, native: bool | None = None, threads: int = 0, trim: bool = False, device: int | None = None) -> ReadsSoA:
    """Decode ``path`` into a ReadsSoA (BAM order).  ``intervals`` = [(chrom, start, end)]: keep only reads whose
    reference span touches a target interval (the only reads a pileup over those targets can see).  With intervals and a
    .bai beside the BAM that is not older than it (``find_index``), only the index chunks the intervals need are read and
    inflated; the result is the same as that of a whole-file decode.

    ``native``: True = require libsmc_bamio.so, False = Python walker, None = native when built.
    ``trim``: store only each read's target window (ReadsSoA.store_lo / store_len): what the calling path uploads.
    ``device``: None = decode on the host; a GPU index = inflate and decode on that GPU (libsmc_b200: smc_decode_bam), with the
    same result; a file the GPU cannot take is decoded on the host with a warning line."""
    index = find_index(path) if intervals else None
    if device is not None:
        from . import _bamio
        return _bamio.read_bam_device(path, intervals, int(device), threads, trim, index=index)
    if native is not False:
        try:
            from . import _bamio
            return _bamio.read_bam_native(path, intervals, threads, trim, index=index)
        except ImportError:
            if native:
                raise
    if index is not None:
        with open(path, "rb") as fh:
            _text, refs = read_header_blocks(fh)
        names = [n for n, _ in refs]
        raw, first = read_chunks(path, bai_chunks(read_bai(index, len(refs)), names, intervals), index), 0
    else:
        with open(path, "rb") as fh:
            raw = bgzf_decompress(fh.read())
        _text, refs, first = parse_header(raw)
    soa = decode_records_py(raw, first, [n for n, _ in refs], intervals)
    return soa.trim_to_targets(intervals) if (trim and intervals) else soa


# ------------------------------------------------------------------------------------------------------------------
# writer (tests, examples): ReadsSoA -> BAM
# ------------------------------------------------------------------------------------------------------------------
def _reg2bin(beg, end):
    end -= 1
    if beg >> 14 == end >> 14: return ((1 << 15) - 1) // 7 + (beg >> 14)
    if beg >> 17 == end >> 17: return ((1 << 12) - 1) // 7 + (beg >> 17)
    if beg >> 20 == end >> 20: return ((1 << 9) - 1) // 7 + (beg >> 20)
    if beg >> 23 == end >> 23: return ((1 << 6) - 1) // 7 + (beg >> 23)
    if beg >> 26 == end >> 26: return ((1 << 3) - 1) // 7 + (beg >> 26)
    return 0


def write_bam(path: str, soa: ReadsSoA, ref_lengths: dict, qname_fn=None, nm_type: str = "C", extra_tags: bytes = b"",
              level: int = 1, index: bool = False, block: int = 0xff00):
    """Write ``soa`` as a coordinate-sorted BAM.  Read names are ``<readid>:<barcode>:<x>`` so that the identity parse of
    smCounter.py:319-325 round-trips; ``qname_fn(i, frag_id, barcode)`` overrides the name.  ``index``: also write
    ``<path>.bai``.  ``block``: inflated bytes per BGZF block."""
    from .soa import umi_string
    text = "@HD\tVN:1.4\tSO:coordinate\n" + "".join("@SQ\tSN:%s\tLN:%d\n" % (c, ref_lengths[c]) for c in soa.chroms)
    parts = [b"BAM\x01", struct.pack("<i", len(text)), text.encode(), struct.pack("<i", len(soa.chroms))]
    for c in soa.chroms:
        parts.append(struct.pack("<i", len(c) + 1) + c.encode() + b"\x00" + struct.pack("<i", ref_lengths[c]))
    ends = soa.ref_end()
    nm_fmt = {"C": "<B", "c": "<b", "S": "<H", "s": "<h", "I": "<I", "i": "<i"}[nm_type]
    off = sum(len(x) for x in parts)
    recs = []                                   # (ref_id, pos, end, bin, flag, inflated offset of the record, of its end)
    for i in range(soa.n):
        bc = umi_string(int(soa.umi[i]), soa.umi_names)
        fid = int(soa.frag_id[i])
        qn = (qname_fn(i, fid, bc) if qname_fn else "M1:F%d:%s:%d" % (fid, bc, 1 + ((int(soa.flag[i]) >> 7) & 1))).encode() + b"\x00"
        L = int(soa.l_seq[i]); nc = int(soa.n_cigar[i])
        so, qo, co = int(soa.seq_off[i]), int(soa.qual_off[i]), int(soa.cigar_off[i])
        pos = int(soa.pos[i])
        end = max(int(ends[i]), pos + 1)
        b = _reg2bin(pos, end)
        body = struct.pack("<iiBBHHHiiii", int(soa.ref_id[i]), pos, len(qn), int(soa.mapq[i]), b, nc, int(soa.flag[i]), L, -1, -1, 0)
        body += qn + soa.cigar[co:co + nc].astype("<u4").tobytes() + soa.seq[so:so + (L + 1) // 2].tobytes() + \
            soa.qual[qo:qo + L].tobytes() + extra_tags + b"NM" + nm_type.encode() + struct.pack(nm_fmt, int(soa.nm[i]))
        parts.append(struct.pack("<i", len(body)) + body)
        recs.append((int(soa.ref_id[i]), pos, end, b, int(soa.flag[i]), off, off + len(parts[-1])))
        off += len(parts[-1])
    blocks = _bgzf_block_list(b"".join(parts), level, block)
    with open(path, "wb") as fh:
        fh.write(b"".join(blocks + [_BGZF_EOF]))
    if index:
        coff = np.concatenate(([0], np.cumsum([len(x) for x in blocks], dtype=np.int64))).tolist()
        voff = lambda p: (coff[p // block] << 16) | (p % block)      # p == len(raw): the EOF block, offset 0
        with open(path + ".bai", "wb") as fh:
            fh.write(bai_bytes(recs, len(soa.chroms), voff))


def bai_bytes(recs, n_ref: int, voff) -> bytes:
    """The .bai of coordinate-sorted records ``recs`` = [(ref_id, pos, end, bin, flag, start, stop)] (start / stop: inflated
    offsets, ``voff`` turns them into virtual offsets): one chunk per run of consecutive records in the same bin, linear-index
    entries for every 16 kbp window a record overlaps (0 for windows no record overlaps), the pseudo-bin, n_no_coor."""
    per = [dict(bins={}, lin=[], first=None, last=None, mapped=0, unmapped=0) for _ in range(n_ref)]
    n_no_coor, prev = 0, None
    for (rid, pos, end, b, flag, start, stop) in recs:
        if rid < 0:
            n_no_coor += 1
            continue
        R = per[rid]
        vb, ve = voff(start), voff(stop)
        if prev == (rid, b):
            R["bins"][b][-1][1] = ve
        else:
            R["bins"].setdefault(b, []).append([vb, ve])
        prev = (rid, b)
        lin = R["lin"]
        for w in range(pos >> 14, ((end - 1) >> 14) + 1):
            if w >= len(lin):
                lin.extend([0] * (w + 1 - len(lin)))
            if lin[w] == 0:
                lin[w] = vb
        if R["first"] is None:
            R["first"] = vb
        R["last"] = ve
        R["unmapped" if flag & 0x4 else "mapped"] += 1
    out = [b"BAI\x01", struct.pack("<i", n_ref)]
    for R in per:
        bins = sorted(R["bins"].items())
        out.append(struct.pack("<i", len(bins) + (R["first"] is not None)))
        for b, chunks in bins:
            out.append(struct.pack("<Ii", b, len(chunks)) + b"".join(struct.pack("<QQ", x, y) for x, y in chunks))
        if R["first"] is not None:
            out.append(struct.pack("<IiQQQQ", _PSEUDO_BIN, 2, R["first"], R["last"], R["mapped"], R["unmapped"]))
        out.append(struct.pack("<i", len(R["lin"])) + b"".join(struct.pack("<Q", x) for x in R["lin"]))
    out.append(struct.pack("<Q", n_no_coor))
    return b"".join(out)
