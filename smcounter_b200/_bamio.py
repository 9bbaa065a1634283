"""ctypes binding of libsmc_bamio.so (include/smc_bamio.h): threaded BGZF inflate + BAM record walk in C++."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from .soa import ReadsSoA

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsmc_bamio.so")
EXPORTS = ("smc_bam_set_trim", "smc_bam_open", "smc_bam_open_indexed", "smc_bam_close", "smc_bam_last_error", "smc_bam_n_refs", "smc_bam_ref_name", "smc_bam_ref_length",
           "smc_bam_decode", "smc_bam_dict_umi", "smc_bam_inflate_raw", "smc_rows_emit", "smc_rows_free", "smc_soa_qual_hist", "smc_soa_ref_end", "smc_soa_order_stats", "smc_soa_pack_begin", "smc_soa_pack_fill",
           "smc_soa_pack_end")
_vp = C.c_void_p


class smc_bam_reads(C.Structure):
    _fields_ = [("n_reads", C.c_int64), ("ref_id", _vp), ("pos", _vp), ("flag", _vp), ("mapq", _vp), ("nm", _vp), ("l_seq", _vp),
                ("seq_off", _vp), ("qual_off", _vp), ("cigar_off", _vp), ("n_cigar", _vp), ("umi", _vp), ("frag_id", _vp),
                ("seq", _vp), ("seq_bytes", C.c_int64), ("qual", _vp), ("qual_bytes", C.c_int64), ("cigar", _vp),
                ("n_cigar_words", C.c_int64), ("n_dict_umis", C.c_int64), ("store_lo", _vp), ("store_len", _vp), ("qual_hist", _vp)]


class smc_rows_in(C.Structure):               # include/smc_rows.h
    _fields_ = [("n_loci", C.c_int64), ("n_rows", C.c_int64), ("order", _vp), ("ref_id", _vp), ("pos0", _vp), ("ref_base", _vp),
                ("n_chroms", C.c_int32), ("chroms", C.POINTER(C.c_char_p)), ("loc", _vp), ("cnt", _vp), ("pi", _vp), ("alt_allele", _vp),
                ("second_allele", _vp), ("fl1", _vp), ("fl2", _vp), ("biallelic", _vp), ("n_dyn", C.c_int64), ("dyn_cnt", _vp), ("dyn_pi", _vp),
                ("dyn_names", _vp), ("dyn_name_off", _vp), ("hp1", _vp), ("hp2", _vp), ("finalize", C.c_int32), ("threshold", C.c_int32),
                ("n_trf", C.c_int64), ("trf_chrom", _vp), ("trf_lo", _vp), ("trf_hi", _vp), ("n_rm", C.c_int64), ("rm_chrom", _vp),
                ("rm_lo", _vp), ("rm_hi", _vp), ("rm_tags", _vp), ("rm_tag_off", _vp), ("threads", C.c_int32), ("reserved0", C.c_int32)]


class smc_rows_out(C.Structure):
    _fields_ = [("all", _vp), ("all_off", _vp), ("cut", _vp), ("cut_off", _vp), ("vcf", _vp), ("vcf_off", _vp), ("bad_row", C.c_int64),
                ("bad_status", C.c_uint32)]


class smc_soa_view(C.Structure):             # include/smc_soa.h
    _fields_ = [("n_reads", C.c_int64), ("ref_id", _vp), ("pos", _vp), ("flag", _vp), ("mapq", _vp), ("nm", _vp), ("l_seq", _vp),
                ("seq_off", _vp), ("qual_off", _vp), ("cigar_off", _vp), ("n_cigar", _vp), ("umi", _vp), ("frag_id", _vp),
                ("seq", _vp), ("qual", _vp), ("cigar", _vp), ("store_lo", _vp), ("store_len", _vp)]


class smc_soa_pack_opts(C.Structure):
    _fields_ = [("scalar_bits", C.c_int32), ("qual_bits", C.c_int32), ("seq_bits", C.c_int32), ("threads", C.c_int32), ("ref_id_bits", C.c_int32),
                ("umi_bits", C.c_int32), ("code_of", C.c_uint8 * 256)]


class smc_soa_pack_sizes(C.Structure):
    _fields_ = [("n_reads", C.c_int64), ("seq_bytes", C.c_int64), ("qual_bytes", C.c_int64), ("n_cigar_words", C.c_int64)]


class smc_soa_pack_bufs(C.Structure):
    _fields_ = [("ref_id", _vp), ("pos", _vp), ("flag", _vp), ("mapq", _vp), ("nm", _vp), ("l_seq", _vp), ("store_lo", _vp), ("store_len", _vp),
                ("n_cigar", _vp), ("umi", _vp), ("frag_id", _vp), ("seq", _vp), ("qual", _vp), ("cigar", _vp), ("seq_poff", _vp)]


class smc_soa_pack_exc(C.Structure):
    _fields_ = [("n", C.c_int64), ("read", _vp), ("pos", _vp), ("nib", _vp)]


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("libsmc_bamio.so is not built (%s); run `python -m smcounter_b200.build`" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    lib.smc_bam_open.argtypes = [C.c_char_p, C.c_int, C.POINTER(_vp)]
    lib.smc_bam_open.restype = C.c_int
    lib.smc_bam_open_indexed.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.POINTER(_vp)]
    lib.smc_bam_open_indexed.restype = C.c_int
    lib.smc_bam_close.argtypes = [_vp]
    lib.smc_bam_close.restype = None
    lib.smc_bam_set_trim.argtypes = [_vp, C.c_int]
    lib.smc_bam_set_trim.restype = None
    lib.smc_bam_last_error.argtypes = [_vp]
    lib.smc_bam_last_error.restype = C.c_char_p
    lib.smc_bam_n_refs.argtypes = [_vp]
    lib.smc_bam_n_refs.restype = C.c_int
    lib.smc_bam_ref_name.argtypes = [_vp, C.c_int]
    lib.smc_bam_ref_name.restype = C.c_char_p
    lib.smc_bam_ref_length.argtypes = [_vp, C.c_int]
    lib.smc_bam_ref_length.restype = C.c_int64
    lib.smc_bam_decode.argtypes = [_vp, C.c_int64, _vp, _vp, _vp, C.POINTER(smc_bam_reads)]
    lib.smc_bam_decode.restype = C.c_int
    lib.smc_bam_dict_umi.argtypes = [_vp, C.c_int64]
    lib.smc_bam_dict_umi.restype = C.c_char_p
    lib.smc_bam_inflate_raw.argtypes = [_vp, C.c_int64, _vp, C.c_int64]
    lib.smc_bam_inflate_raw.restype = C.c_int
    lib.smc_rows_emit.argtypes = [C.POINTER(smc_rows_in), C.POINTER(smc_rows_out)]
    lib.smc_rows_emit.restype = C.c_int
    lib.smc_rows_free.argtypes = [C.POINTER(smc_rows_out)]
    lib.smc_rows_free.restype = None
    lib.smc_soa_qual_hist.argtypes = [C.POINTER(smc_soa_view), C.c_int, _vp]
    lib.smc_soa_qual_hist.restype = C.c_int
    lib.smc_soa_ref_end.argtypes = [C.POINTER(smc_soa_view), C.c_int, _vp]
    lib.smc_soa_ref_end.restype = C.c_int
    lib.smc_soa_order_stats.argtypes = [C.POINTER(smc_soa_view), C.c_int, _vp, _vp]
    lib.smc_soa_order_stats.restype = C.c_int
    lib.smc_soa_pack_begin.argtypes = [C.POINTER(smc_soa_view), _vp, C.c_int64, C.POINTER(smc_soa_pack_opts), C.POINTER(_vp), C.POINTER(smc_soa_pack_sizes)]
    lib.smc_soa_pack_begin.restype = C.c_int
    lib.smc_soa_pack_fill.argtypes = [_vp, C.POINTER(smc_soa_pack_bufs), C.POINTER(smc_soa_pack_exc)]
    lib.smc_soa_pack_fill.restype = C.c_int
    lib.smc_soa_pack_end.argtypes = [_vp]
    lib.smc_soa_pack_end.restype = None
    _lib = lib
    return lib


class _Handle:
    """Owns an smc_bam handle; closed when the last array that views its buffers is gone."""

    def __init__(self, lib, h):
        self.lib, self.h = lib, h

    def close(self):
        if self.h:
            self.lib.smc_bam_close(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _arr(ptr, n, dtype, owner):
    """numpy view of a decoder buffer (no copy): the ctypes buffer the array is based on keeps ``owner`` alive."""
    n = int(n)
    if n == 0 or not ptr:
        return np.zeros(0, dtype=dtype)
    buf = (C.c_char * (n * np.dtype(dtype).itemsize)).from_address(ptr)
    buf._smc_owner = owner
    return np.frombuffer(buf, dtype=dtype, count=n)


E_INDEX = -3                       # include/smc_bamio.h: the index is malformed or does not fit the BAM


def _raise(rc, msg):
    raise (IOError if rc == E_INDEX else ValueError)(msg.decode())


def read_bam_native(path: str, intervals=None, threads: int = 0, trim: bool = False, index: str | None = None) -> ReadsSoA:
    """``index``: path of the BAM's .bai; with intervals, only the index chunks they need are read and inflated."""
    lib = load()
    h = _vp()
    if index is not None:
        rc = lib.smc_bam_open_indexed(os.fsencode(path), os.fsencode(index), int(threads), C.byref(h))
    else:
        rc = lib.smc_bam_open(os.fsencode(path), int(threads), C.byref(h))
    if rc != 0:
        _raise(rc, lib.smc_bam_last_error(None))
    owner = _Handle(lib, h)
    ok = False
    try:
        chroms = [lib.smc_bam_ref_name(h, i).decode() for i in range(lib.smc_bam_n_refs(h))]
        cidx = {c: i for i, c in enumerate(chroms)}
        ivs = [(cidx[c], s, e) for (c, s, e) in (intervals or ()) if c in cidx and e > s]
        iv_ref = np.asarray([v[0] for v in ivs], dtype=np.int32)
        iv_s = np.asarray([v[1] for v in ivs], dtype=np.int32)
        iv_e = np.asarray([v[2] for v in ivs], dtype=np.int32)
        out = smc_bam_reads()
        if intervals is not None and not ivs:
            n_iv, args = 1, (np.asarray([-1], np.int32), np.zeros(1, np.int32), np.zeros(1, np.int32))   # nothing can match
        else:
            n_iv, args = len(ivs), (iv_ref, iv_s, iv_e)
        lib.smc_bam_set_trim(h, 1 if (trim and ivs) else 0)
        rc = lib.smc_bam_decode(h, n_iv, args[0].ctypes.data, args[1].ctypes.data, args[2].ctypes.data, C.byref(out))
        if rc != 0:
            _raise(rc, lib.smc_bam_last_error(h))
        n = out.n_reads
        A = lambda ptr, count, dtype: _arr(ptr, count, dtype, owner)
        umi = A(out.umi, n, np.uint64)
        names = {}
        for i in range(out.n_dict_umis):
            names[(1 << 63) | i] = lib.smc_bam_dict_umi(h, i).decode()
        # 2-bit packed codes decode to their barcode on demand (soa.umi_string); only the dictionary-coded ones need a name
        soa = ReadsSoA(
            ref_id=A(out.ref_id, n, np.int32), pos=A(out.pos, n, np.int32), flag=A(out.flag, n, np.uint16),
            mapq=A(out.mapq, n, np.uint8), nm=A(out.nm, n, np.int32), l_seq=A(out.l_seq, n, np.int32),
            seq_off=A(out.seq_off, n, np.int64), qual_off=A(out.qual_off, n, np.int64), cigar_off=A(out.cigar_off, n, np.int64),
            n_cigar=A(out.n_cigar, n, np.uint16), umi=umi, frag_id=A(out.frag_id, n, np.uint32),
            seq=A(out.seq, out.seq_bytes, np.uint8), qual=A(out.qual, out.qual_bytes, np.uint8),
            cigar=A(out.cigar, out.n_cigar_words, np.uint32), chroms=chroms, umi_names=names, packed=True,
            store_lo=A(out.store_lo, n, np.int32) if out.store_lo else None,
            store_len=A(out.store_len, n, np.int32) if out.store_len else None)
        if out.qual_hist:                   # counted during the decode: the upload codebook needs no pass of its own
            soa.__dict__["_qual_hist"] = np.frombuffer((C.c_uint64 * 256).from_address(out.qual_hist), dtype=np.uint64).copy()
        ok = True
        return soa
    finally:
        if not ok:
            owner.close()


# ------------------------------------------------------------------------------------------------------------
# include/smc_soa.h: the reads of a batch, gathered and written in the compact wire encodings in one native pass
def _view(r: ReadsSoA) -> smc_soa_view:
    v = smc_soa_view()
    v.n_reads = r.n
    for f in ("ref_id", "pos", "flag", "mapq", "nm", "l_seq", "seq_off", "qual_off", "cigar_off", "n_cigar", "umi", "frag_id", "seq", "qual", "cigar"):
        a = getattr(r, f)
        assert a.flags["C_CONTIGUOUS"]
        setattr(v, f, a.ctypes.data)
    if r.store_lo is not None:
        v.store_lo, v.store_len = r.store_lo.ctypes.data, r.store_len.ctypes.data
    return v


def ref_end_native(reads: ReadsSoA, threads: int = 0) -> np.ndarray:
    """ReadsSoA.ref_end() by one threaded native pass over the CIGARs."""
    out = np.empty(reads.n, np.int64)
    v = _view(reads)
    rc = load().smc_soa_ref_end(C.byref(v), threads, out.ctypes.data)
    if rc:
        raise RuntimeError("smc_soa_ref_end failed (%d)" % rc)
    return out


def order_stats_native(reads: ReadsSoA, threads: int = 0):
    """(ref_end, in BAM coordinate order?, longest reference span) by one threaded native pass."""
    out = np.empty(reads.n, np.int64)
    st = np.zeros(2, np.int64)
    v = _view(reads)
    rc = load().smc_soa_order_stats(C.byref(v), threads, out.ctypes.data, st.ctypes.data)
    if rc:
        raise RuntimeError("smc_soa_order_stats failed (%d)" % rc)
    return out, bool(st[0]), int(st[1])


def upload_codebook(reads: ReadsSoA, threads: int = 0) -> dict:
    """What every batch of ``reads`` is packed with (memoised on the SoA): 16-bit scalars when every value fits, the
    quality codebook (2 / 4 bits when at most 4 / 16 distinct phred values occur in the whole file)."""
    memo = reads.__dict__.get("_upload_codebook")
    if memo is not None:
        return memo
    lib = load()
    hist = reads.__dict__.get("_qual_hist")
    if hist is None:
        hist = np.zeros(256, np.uint64)
        v = _view(reads)
        rc = lib.smc_soa_qual_hist(C.byref(v), threads, hist.ctypes.data)
        if rc:
            raise RuntimeError("smc_soa_qual_hist failed (%d)" % rc)
    present = np.flatnonzero(hist)
    bits = 2 if len(present) <= 4 else 4 if len(present) <= 16 else 8
    lut = code_of = None
    if bits != 8:
        lut = np.zeros(1 << bits, np.uint8)
        lut[:len(present)] = present
        code_of = np.full(256, 0xFF, np.uint8)
        code_of[present] = np.arange(len(present), dtype=np.uint8)
    scal = [reads.nm, reads.l_seq] + ([] if reads.store_lo is None else [reads.store_lo, reads.store_len])
    top = max([0] + [int(a.max()) for a in scal if len(a)])
    low = min([0] + [int(a.min()) for a in scal if len(a)])
    sbits = 32 if (low < 0 or top >= 65536) else 16 if top >= 256 else 8
    ref8 = bool(reads.n) and int(reads.ref_id.min()) >= 0 and int(reads.ref_id.max()) < 256
    umi32 = bool(reads.n) and int(reads.umi.max()) < (1 << 32)
    memo = dict(scalar_bits=sbits, qual_bits=bits, qual_lut=lut, code_of=code_of, ref_id_bits=8 if ref8 else 32, umi_bits=32 if umi32 else 64)
    reads.__dict__["_upload_codebook"] = memo
    return memo


def pack_upload(reads: ReadsSoA, idx=None, alloc=None, seq_bits: int = 2, threads: int = 0) -> ReadsSoA:
    """The reads ``idx`` (ascending; None = all) of a plain SoA as a compact upload SoA (ReadsSoA.compact() of
    ReadsSoA.select(idx), bit for bit) made by one threaded native pass.  ``alloc(nbytes) -> uint8 array`` supplies the
    output buffers (a pinned arena: caller.PinnedArena.take); default: ordinary numpy memory."""
    if reads.qual_bits != 8 or reads.scalar_bits != 32 or reads.seq_bits != 4:
        raise ValueError("pack_upload needs a plain SoA")
    lib = load()
    cb = upload_codebook(reads, threads)
    alloc = alloc or (lambda nbytes: np.empty(nbytes, np.uint8))
    take = lambda count, dt: alloc(max(int(count), 1) * np.dtype(dt).itemsize).view(dt)[:int(count)]
    o = smc_soa_pack_opts()
    o.scalar_bits, o.qual_bits, o.seq_bits, o.threads = cb["scalar_bits"], cb["qual_bits"], seq_bits, threads
    o.ref_id_bits, o.umi_bits = cb["ref_id_bits"], cb["umi_bits"]
    if cb["code_of"] is not None:
        C.memmove(o.code_of, cb["code_of"].ctypes.data, 256)
    v = _view(reads)
    if idx is not None:
        idx = np.ascontiguousarray(idx, dtype=np.int64)
    h, sz = _vp(), smc_soa_pack_sizes()
    rc = lib.smc_soa_pack_begin(C.byref(v), None if idx is None else idx.ctypes.data, 0 if idx is None else len(idx), C.byref(o), C.byref(h), C.byref(sz))
    if rc:
        raise RuntimeError("smc_soa_pack_begin failed (%d)" % rc)
    try:
        n = int(sz.n_reads)
        sdt = {8: np.uint8, 16: np.uint16, 32: np.int32}[cb["scalar_bits"]]
        out = dict(ref_id=take(n, np.uint8 if cb["ref_id_bits"] == 8 else np.int32), pos=take(n, np.int32), flag=take(n, np.uint16),
                   mapq=take(n, np.uint8), nm=take(n, sdt), l_seq=take(n, sdt), n_cigar=take(n, np.uint16),
                   umi=take(n, np.uint32 if cb["umi_bits"] == 32 else np.uint64), frag_id=take(n, np.uint32),
                   seq=take(sz.seq_bytes, np.uint8), qual=take(sz.qual_bytes, np.uint8), cigar=take(sz.n_cigar_words, np.uint32))
        if reads.store_lo is not None:
            out["store_lo"], out["store_len"] = take(n, sdt), take(n, sdt)
        poff = np.empty(n + 1, np.int64)
        b = smc_soa_pack_bufs()
        for f, a in out.items():
            setattr(b, f, a.ctypes.data)
        b.seq_poff = poff.ctypes.data
        ex = smc_soa_pack_exc()
        rc = lib.smc_soa_pack_fill(h, C.byref(b), C.byref(ex))
        if rc:
            raise RuntimeError("smc_soa_pack_fill failed (%d): a scalar above 65535 or a quality outside the codebook" % rc)
        exc = None
        if seq_bits == 2:
            ne = int(ex.n)
            exc = (take(ne, np.uint32), take(ne, np.uint32), take(ne, np.uint8))
            if ne:
                C.memmove(exc[0].ctypes.data, ex.read, 4 * ne); C.memmove(exc[1].ctypes.data, ex.pos, 4 * ne); C.memmove(exc[2].ctypes.data, ex.nib, ne)
    finally:
        lib.smc_soa_pack_end(h)
    zero = np.zeros(0, np.int64)
    res = ReadsSoA(seq_off=zero, qual_off=zero, cigar_off=zero, chroms=reads.chroms, umi_names=reads.umi_names, packed=True,
                   scalar_bits=cb["scalar_bits"], qual_bits=cb["qual_bits"], qual_lut=cb["qual_lut"], seq_bits=seq_bits, seq_exc=exc,
                   store_lo=out.get("store_lo"), store_len=out.get("store_len"),
                   **{f: out[f] for f in ("ref_id", "pos", "flag", "mapq", "nm", "l_seq", "n_cigar", "umi", "frag_id", "seq", "qual", "cigar")})
    if seq_bits == 2:
        res.__dict__["_compact_memo"] = (poff, (exc[0].astype(np.uint64) << np.uint64(32)) | exc[1].astype(np.uint64))
    else:
        res.seq_off = poff[:-1]
    return res
