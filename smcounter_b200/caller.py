"""Host side of the hot path: one batched call per GPU into libsmc_b200.so, replacing the reference's
``Pool.apply_async(vc_wrapper, ...)`` fan-out (smCounter.py:683-685) and the body of ``vc()`` (:274-600).

``GpuCaller.call(reads, loci)`` returns ``LocusResults`` (flat numpy arrays, one entry per target locus);
``smcounter_b200.rows.format_rows`` turns those into the reference's 45-column rows.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _ffi
from .soa import Loci, ReadsSoA


@dataclass
class VcParams:
    """The parameters of vc() (smCounter.py:274) with the CLI defaults of smCounter.py:619-633."""
    mtDepth: int
    rpb: float
    minBQ: int = 20
    minMQ: int = 30
    hpLen: int = 10
    mismatchThr: float = 6.0
    mtDrop: int = 0
    maxMT: int = 0
    primerDist: int = 2
    fisherLegacy: int = 0      # 0: scipy >= 1.7 fisher_exact semantics (what the oracle's scipy does); 1: scipy <= 1.6 (epsilon = 1 - 1e-4)

    @property
    def ds(self) -> int:
        """Down-sampling cap (smCounter.py:486); Python-2 round() is half away from zero, exact for 2*int."""
        return self.maxMT if self.maxMT > 0 else int(2 * self.mtDepth)


def _alloc(shape, dtype, pinned):
    if pinned:
        import torch
        t = torch.empty(int(np.prod(shape)) * np.dtype(dtype).itemsize, dtype=torch.uint8, pin_memory=True)
        return t.numpy().view(dtype).reshape(shape)
    return np.empty(shape, dtype=dtype)


class PinnedArena:
    """Page-locked host memory (smc_host_alloc) handed out in 256-byte aligned pieces and recycled batch after batch:
    ``take(nbytes)`` until ``reset()``.  What _bamio.pack_upload writes a batch into, so that smc_call_batch's copies
    run as DMA at the link rate.  Slabs only grow; ``close()`` frees them."""

    def __init__(self, first_bytes: int = 64 << 20):
        self.lib = _ffi.load()
        self.slabs = []             # (address, size, uint8 view)
        self.cur, self.off = 0, 0
        self.first = int(first_bytes)

    def _new_slab(self, nbytes):
        p = C.c_void_p()
        rc = self.lib.smc_host_alloc(nbytes, C.byref(p))
        if rc != 0 or not p.value:
            raise MemoryError("smc_host_alloc(%d) failed (%d)" % (nbytes, rc))
        view = np.frombuffer((C.c_uint8 * nbytes).from_address(p.value), dtype=np.uint8)
        self.slabs.append((p.value, nbytes, view))

    def take(self, nbytes: int) -> np.ndarray:
        nbytes = max(int(nbytes), 1)
        need = (nbytes + 255) & ~255
        while True:
            if self.cur < len(self.slabs):
                _, size, view = self.slabs[self.cur]
                if self.off + need <= size:
                    out = view[self.off:self.off + nbytes]
                    self.off += need
                    return out
                self.cur, self.off = self.cur + 1, 0
                continue
            last = self.slabs[-1][1] if self.slabs else self.first // 2
            self._new_slab(max(2 * last, need))

    def reset(self):
        self.cur, self.off = 0, 0

    def close(self):
        for (addr, _, _) in self.slabs:
            self.lib.smc_host_free(addr)
        self.slabs = []
        self.reset()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class LocusResults:
    """Per-locus outputs of the device path (include/smc_b200.h: smc_out)."""

    def __init__(self, n_loci: int, dyn_capacity: int, pinned: bool = False):
        self.n_loci = n_loci
        self.dyn_capacity = dyn_capacity
        n = max(n_loci, 1)
        d = max(dyn_capacity, 1)
        self.loc = _alloc((_ffi.SMC_NLOC, n), np.int32, pinned)
        self.cnt = _alloc((_ffi.SMC_NFIXED, _ffi.SMC_NCNT, n), np.int32, pinned)
        self.pi = _alloc((_ffi.SMC_NFIXED, n), np.float64, pinned)
        self.max_allele = _alloc((n,), np.int32, pinned)
        self.second_allele = _alloc((n,), np.int32, pinned)
        self.alt_allele = _alloc((n,), np.int32, pinned)
        self.alt_pi = _alloc((n,), np.float64, pinned)
        self.second_pi = _alloc((n,), np.float64, pinned)
        self.fl1 = _alloc((n,), np.uint32, pinned)
        self.fl2 = _alloc((n,), np.uint32, pinned)
        self.biallelic = _alloc((n,), np.uint8, pinned)
        self.fisher_p = _alloc((2, 4, n), np.float64, pinned)
        self.fisher_or = _alloc((2, 4, n), np.float64, pinned)
        self.dyn_locus = _alloc((d,), np.int32, pinned)
        self.dyn_kind = _alloc((d,), np.uint8, pinned)
        self.dyn_site = _alloc((d,), np.uint8, pinned)
        self.dyn_len = _alloc((d,), np.int32, pinned)
        self.dyn_rep_read = _alloc((d,), np.uint32, pinned)
        self.dyn_rep_qpos = _alloc((d,), np.int32, pinned)
        self.dyn_iskey = _alloc((d,), np.uint8, pinned)
        self.dyn_cnt = _alloc((d, _ffi.SMC_NCNT), np.int32, pinned)
        self.dyn_pi = _alloc((d,), np.float64, pinned)
        self.dyn_first = _alloc((n + 1,), np.int64, pinned)
        self.n_dyn = 0

    def as_struct(self) -> _ffi.smc_out:
        p = _ffi.ptr
        o = _ffi.smc_out()
        o.n_loci = self.n_loci
        o.loc, o.cnt, o.pi = p(self.loc), p(self.cnt), p(self.pi)
        o.max_allele, o.second_allele, o.alt_allele = p(self.max_allele), p(self.second_allele), p(self.alt_allele)
        o.alt_pi, o.second_pi, o.fl1, o.fl2, o.biallelic = p(self.alt_pi), p(self.second_pi), p(self.fl1), p(self.fl2), p(self.biallelic)
        o.fisher_p, o.fisher_or = p(self.fisher_p), p(self.fisher_or)
        o.dyn_capacity = self.dyn_capacity
        o.n_dyn = 0
        o.dyn_locus, o.dyn_kind, o.dyn_site, o.dyn_len = p(self.dyn_locus), p(self.dyn_kind), p(self.dyn_site), p(self.dyn_len)
        o.dyn_rep_read, o.dyn_rep_qpos, o.dyn_iskey = p(self.dyn_rep_read), p(self.dyn_rep_qpos), p(self.dyn_iskey)
        o.dyn_cnt, o.dyn_pi, o.dyn_first = p(self.dyn_cnt), p(self.dyn_pi), p(self.dyn_first)
        return o

    def nbytes(self) -> int:
        return sum(v.nbytes for v in self.__dict__.values() if isinstance(v, np.ndarray))


class UmiKeep:
    """Down-sampling mask (smCounter.py:496-500): {locus index -> iterable of kept barcode codes}."""

    def __init__(self, mapping: dict):
        items = sorted((int(k), np.sort(np.asarray(list(v), dtype=np.uint64))) for k, v in mapping.items())
        self.locus = np.asarray([k for k, _ in items], dtype=np.int64)
        self.off = np.zeros(len(items) + 1, dtype=np.int64)
        for i, (_, v) in enumerate(items):
            self.off[i + 1] = self.off[i] + len(v)
        self.umi = np.concatenate([v for _, v in items]) if items else np.zeros(0, np.uint64)

    def as_struct(self) -> _ffi.smc_umi_keep:
        k = _ffi.smc_umi_keep()
        k.n_loci = len(self.locus)
        k.locus, k.off, k.umi = _ffi.ptr(self.locus), _ffi.ptr(self.off), _ffi.ptr(self.umi)
        return k


class GpuCaller:
    """One context per GPU (not thread-safe per context; ctypes releases the GIL during calls).

    ``device_downsample``: draw the reference's down-sampling sample on the device inside every call (smc_set_downsample), so
    that no locus comes back flagged ST_NEED_DOWNSAMPLE; dictionary-coded barcodes need their hashes (set_barcode_hashes)."""

    def __init__(self, params: VcParams, device: int = 0, device_downsample: bool = False):
        self.lib = _ffi.load()
        self.params = params
        p = _ffi.smc_params(params.minBQ, params.minMQ, params.mtDepth, params.mtDrop, params.maxMT, params.primerDist,
                            float(params.rpb), float(params.mismatchThr), int(params.fisherLegacy), 0)
        h = C.c_void_p()
        rc = self.lib.smc_ctx_create(int(device), C.byref(p), C.byref(h))
        if rc != 0:
            raise RuntimeError("smc_ctx_create failed (%d): %s" % (rc, self.lib.smc_last_error(None).decode()))
        self.h = h
        self._keepalive = None
        if device_downsample:
            rc = self.lib.smc_set_downsample(self.h, _ffi.DS_DEVICE)
            if rc != 0:
                raise self._err("smc_set_downsample", rc)

    def close(self):
        if getattr(self, "h", None):
            self.lib.smc_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _err(self, what, rc, loci=None):
        msg = self.lib.smc_last_error(self.h).decode()
        where = ""
        if loci is not None and loci.n:
            where = " in locus range (%d:%d .. %d:%d)" % (loci.ref_id[0], loci.pos0[0] + 1, loci.ref_id[-1], loci.pos0[-1] + 1)
        # mirrors smCounter.py:694 "Exception thrown in vc() at location: ..."
        return RuntimeError("Exception thrown in %s%s: [%d] %s" % (what, where, rc, msg))

    @staticmethod
    def _reads_struct(r: ReadsSoA) -> _ffi.smc_reads_soa:
        p = _ffi.ptr
        s = _ffi.smc_reads_soa()
        s.n_reads = r.n
        s.ref_id, s.pos, s.flag, s.mapq, s.nm, s.l_seq = p(r.ref_id), p(r.pos), p(r.flag), p(r.mapq), p(r.nm), p(r.l_seq)
        s.n_cigar = p(r.n_cigar)
        if getattr(r, "packed", False):        # payload back to back in read order: the library derives the offsets on the device
            s.seq_off = s.qual_off = s.cigar_off = None
        else:
            s.seq_off, s.qual_off, s.cigar_off = p(r.seq_off), p(r.qual_off), p(r.cigar_off)
        s.umi, s.frag_id = p(r.umi), p(r.frag_id)
        s.seq, s.seq_bytes, s.qual, s.qual_bytes = p(r.seq), r.seq.nbytes, p(r.qual), r.qual.nbytes
        s.cigar, s.n_cigar_words = p(r.cigar), r.cigar.shape[0]
        s.store_lo, s.store_len = p(getattr(r, "store_lo", None)), p(getattr(r, "store_len", None))
        s.scalar_bits, s.qual_bits = int(getattr(r, "scalar_bits", 32)), int(getattr(r, "qual_bits", 8))
        s.qual_lut = p(getattr(r, "qual_lut", None))
        s.seq_bits = int(getattr(r, "seq_bits", 4))
        s.ref_id_bits = 8 if r.ref_id.dtype == np.uint8 else 32
        s.umi_bits = 32 if r.umi.dtype == np.uint32 else 64
        exc = getattr(r, "seq_exc", None)
        if s.seq_bits == 2 and exc is not None and len(exc[0]):
            s.n_seq_exc, s.seq_exc_read, s.seq_exc_pos, s.seq_exc_nib = len(exc[0]), p(exc[0]), p(exc[1]), p(exc[2])
        if (s.qual_bits != 8 or s.seq_bits != 4) and not getattr(r, "packed", False):
            raise ValueError("compact qualities / bases need the packed layout")
        return s

    @staticmethod
    def _loci_struct(l: Loci) -> _ffi.smc_loci:
        s = _ffi.smc_loci()
        s.n_loci = l.n
        s.ref_id, s.pos0, s.ref_base = _ffi.ptr(l.ref_id), _ffi.ptr(l.pos0), _ffi.ptr(l.ref_base)
        return s

    def upload(self, reads: ReadsSoA, loci: Loci, keep: UmiKeep | None = None):
        rs, ls = self._reads_struct(reads), self._loci_struct(loci)
        ks = keep.as_struct() if keep is not None else None
        self._keepalive = (reads, loci, keep)
        rc = self.lib.smc_upload(self.h, C.byref(rs), C.byref(ls), C.byref(ks) if ks is not None else None)
        if rc != 0:
            raise self._err("smc_upload", rc, loci)
        self._n_loci = loci.n

    def run(self):
        rc = self.lib.smc_run_resident(self.h)
        if rc != 0:
            raise self._err("smc_run_resident", rc, self._keepalive[1] if self._keepalive else None)

    def download(self, out: LocusResults | None = None) -> LocusResults:
        n_dyn = self.timings()["n_dyn"]
        if out is None or out.n_loci != self._n_loci or out.dyn_capacity < n_dyn:
            out = LocusResults(self._n_loci, max(int(n_dyn), 16))
        o = out.as_struct()
        rc = self.lib.smc_download(self.h, C.byref(o))
        if rc != 0:
            raise self._err("smc_download", rc)
        out.n_dyn = int(o.n_dyn)
        return out

    def call(self, reads: ReadsSoA, loci: Loci, keep: UmiKeep | None = None, out: LocusResults | None = None) -> LocusResults:
        """One ``smc_call_batch``: host buffers in, host buffers out -- the drop-in for the per-locus vc() fan-out
        (smCounter.py:683-685).  The library overlaps the upload of the bases / qualities with the kernels that do not
        need them.  ``out`` is reused when it fits; if the batch has more dynamic-allele rows than ``out`` holds, only the
        download is repeated with a larger buffer (the results stay resident)."""
        if out is None or out.n_loci != loci.n:
            out = LocusResults(loci.n, max(4096, 4 * loci.n))
        rs, ls = self._reads_struct(reads), self._loci_struct(loci)
        ks = keep.as_struct() if keep is not None else None
        self._keepalive = (reads, loci, keep)
        self._n_loci = loci.n
        o = out.as_struct()
        rc = self.lib.smc_call_batch(self.h, C.byref(rs), C.byref(ls), C.byref(ks) if ks is not None else None, C.byref(o))
        if rc == _ffi.SMC_E_LIMIT and int(o.n_dyn) > out.dyn_capacity:
            return self.download(None)
        if rc != 0:
            raise self._err("smc_call_batch", rc, loci)
        out.n_dyn = int(o.n_dyn)
        return out

    def list_barcodes(self, locus_idx):
        """Barcodes of bcDict for the given (ascending) loci of the last batch: (off[n+1], umi codes, first passing read)."""
        locus = np.ascontiguousarray(np.asarray(locus_idx, dtype=np.int64))
        n = int(locus.shape[0])
        off = np.zeros(n + 1, dtype=np.int64)
        rc = self.lib.smc_list_barcodes(self.h, n, _ffi.ptr(locus), _ffi.ptr(off), None, None, 0)
        if rc not in (0, -3):
            raise self._err("smc_list_barcodes", rc)
        total = int(off[n])
        umi = np.zeros(max(total, 1), dtype=np.uint64)
        first = np.zeros(max(total, 1), dtype=np.uint32)
        if total:
            rc = self.lib.smc_list_barcodes(self.h, n, _ffi.ptr(locus), _ffi.ptr(off), _ffi.ptr(umi), _ffi.ptr(first), total)
            if rc != 0:
                raise self._err("smc_list_barcodes", rc)
        return off, umi[:total], first[:total]

    def set_barcode_hashes(self, codes, py2_hashes):
        """The Py2 hash(str) of dictionary-coded barcodes (top bit set) for the following device draws; ``codes`` ascending."""
        c = np.ascontiguousarray(codes, dtype=np.uint64)
        h = np.ascontiguousarray(py2_hashes, dtype=np.int64)
        rc = self.lib.smc_set_barcode_hashes(self.h, len(c), _ffi.ptr(c), _ffi.ptr(h))
        if rc != 0:
            raise self._err("smc_set_barcode_hashes", rc)

    def draw_sample(self, off, codes, seed_pos1, k) -> np.ndarray:
        """random.seed(str(seed_pos1[i])); random.sample(keys in CPython-2 dict order, k[i]) on the device for the key sets
        codes[off[i]:off[i+1]] (insertion order): out[off[i] + j], j < k[i], is the insertion index of the j-th drawn key."""
        off = np.ascontiguousarray(off, dtype=np.int64)
        codes = np.ascontiguousarray(codes, dtype=np.uint64)
        pos = np.ascontiguousarray(seed_pos1, dtype=np.int64)
        k = np.ascontiguousarray(k, dtype=np.int64)
        out = np.full(max(int(off[-1]), 1), -1, dtype=np.int64)
        rc = self.lib.smc_draw_sample(self.h, len(k), _ffi.ptr(off), _ffi.ptr(codes), _ffi.ptr(pos), _ffi.ptr(k), _ffi.ptr(out))
        if rc != 0:
            raise self._err("smc_draw_sample", rc)
        return out[:int(off[-1])]

    def hp_lowcomp(self, hpLen: int, candidates) -> np.ndarray:
        """isHPorLowComp() (smCounter.py:122-177) on the device for ``candidates`` = [(window, pos_in_window, ref, alt)]
        (upper-case ``str``/``bytes``; window = reference[max(0, pos0 - 2*hpLen), min(contig end, pos0 + max(len(ref),
        len(alt)) + 2*hpLen)), see include/smc_b200.h: smc_hp_batch).  Returns uint8 flags: bit 0 homopolymer, bit 1 low complexity."""
        n = len(candidates)
        flags = np.zeros(max(n, 1), dtype=np.uint8)
        if n == 0:
            return flags[:0]
        parts, off = [], 0
        win_off, ref_off, alt_off = np.zeros(n, np.int64), np.zeros(n, np.int64), np.zeros(n, np.int64)
        win_len, win_pos, ref_len, alt_len = (np.zeros(n, np.int32) for _ in range(4))
        for k, (win, wpos, ref, alt) in enumerate(candidates):
            for arr_off, arr_len, sv in ((win_off, win_len, win), (ref_off, ref_len, ref), (alt_off, alt_len, alt)):
                b = sv.encode() if isinstance(sv, str) else bytes(sv)
                arr_off[k], arr_len[k] = off, len(b)
                parts.append(b)
                off += len(b)
            win_pos[k] = wpos
        bases = np.frombuffer(b"".join(parts) or b"\0", dtype=np.uint8)
        hb = _ffi.smc_hp_batch(n, int(hpLen), _ffi.ptr(bases), off, _ffi.ptr(win_off), _ffi.ptr(win_len), _ffi.ptr(win_pos),
                               _ffi.ptr(ref_off), _ffi.ptr(ref_len), _ffi.ptr(alt_off), _ffi.ptr(alt_len))
        rc = self.lib.smc_hp_lowcomp(self.h, C.byref(hb), _ffi.ptr(flags))
        if rc != 0:
            raise self._err("smc_hp_lowcomp", rc)
        return flags[:n]

    def fisher_exact(self, tables):
        """scipy.stats.fisher_exact (two-sided) for an (n, 4) int array of [[a, b], [c, d]] tables on the device: (p, odds)."""
        t = np.ascontiguousarray(tables, dtype=np.int32).reshape(-1, 4)
        p = np.empty(len(t), np.float64); o = np.empty(len(t), np.float64)
        rc = self.lib.smc_fisher_exact(self.h, len(t), t.ctypes.data, p.ctypes.data, o.ctypes.data)
        if rc != 0:
            raise RuntimeError("smc_fisher_exact failed (%d): %s" % (rc, self.lib.smc_last_error(self.h).decode()))
        return p, o

    def timings(self) -> dict:
        t = _ffi.smc_timings()
        self.lib.smc_get_timings(self.h, C.byref(t))
        return {f: getattr(t, f) for f, _ in _ffi.smc_timings._fields_}
