"""ctypes binding of libsmc_b200.so (include/smc_b200.h).  There is no CPU fallback: if the library is not
built, or no CUDA device is present, the constructors raise."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsmc_b200.so")

SMC_NFIXED, SMC_NCNT, SMC_NLOC = 5, 13, 12
SMC_OK, SMC_E_CUDA, SMC_E_ARG, SMC_E_LIMIT, SMC_E_OVERFLOW, SMC_E_STATE, SMC_E_INFLATE, SMC_E_BUDGET = 0, -1, -2, -3, -4, -5, -6, -7
(C_ALLELE, C_FWD, C_REV, C_LOWQ, C_R1LE, C_R1TOT, C_R2LE, C_R2TOT, C_R2PLE, C_CONCORD, C_DISCORD, C_MT,
 C_STRONG) = range(13)
(L_CVG, L_ALLFRAG, L_ALLMT, L_USEDFRAG, L_NBC, L_USEDMT, L_MT3, L_MT5, L_MT7, L_MT10, L_KEYMASK, L_STATUS) = range(12)
ST_ZERO_COVERAGE, ST_NEED_DOWNSAMPLE, ST_UMI_OVERFLOW, ST_BAD_MASK, ST_DOWNSAMPLED = 1, 2, 4, 8, 16
DS_FLAG, DS_DEVICE = 0, 1
K_BASE, K_INS, K_DEL = 0, 1, 2
F_LM, F_LSM, F_DP, F_SB, F_LOWQ, F_R1CP, F_R2CP, F_PRIMERCP = (1 << i for i in range(8))
F_HPGATE, F_EVALUATED = 1 << 16, 1 << 17
A_A, A_C, A_DEL, A_T, A_G = range(5)
FIXED_NAMES = ("A", "C", "DEL", "T", "G")

_vp = C.c_void_p


class smc_params(C.Structure):
    _fields_ = [("minBQ", C.c_int32), ("minMQ", C.c_int32), ("mtDepth", C.c_int32), ("mtDrop", C.c_int32),
                ("maxMT", C.c_int32), ("primerDist", C.c_int32), ("rpb", C.c_double), ("mismatchThr", C.c_double),
                ("fisherLegacy", C.c_int32), ("reserved0", C.c_int32)]


class smc_reads_soa(C.Structure):
    _fields_ = [("n_reads", C.c_int64), ("ref_id", _vp), ("pos", _vp), ("flag", _vp), ("mapq", _vp), ("nm", _vp),
                ("l_seq", _vp), ("seq_off", _vp), ("qual_off", _vp), ("cigar_off", _vp), ("n_cigar", _vp), ("umi", _vp),
                ("frag_id", _vp), ("seq", _vp), ("seq_bytes", C.c_int64), ("qual", _vp), ("qual_bytes", C.c_int64),
                ("cigar", _vp), ("n_cigar_words", C.c_int64), ("store_lo", _vp), ("store_len", _vp),
                ("scalar_bits", C.c_int32), ("qual_bits", C.c_int32), ("qual_lut", _vp),
                ("seq_bits", C.c_int32), ("ref_id_bits", C.c_int32), ("n_seq_exc", C.c_int64), ("seq_exc_read", _vp), ("seq_exc_pos", _vp),
                ("seq_exc_nib", _vp), ("umi_bits", C.c_int32), ("reserved2", C.c_int32)]


class smc_loci(C.Structure):
    _fields_ = [("n_loci", C.c_int64), ("ref_id", _vp), ("pos0", _vp), ("ref_base", _vp)]


class smc_umi_keep(C.Structure):
    _fields_ = [("n_loci", C.c_int64), ("locus", _vp), ("off", _vp), ("umi", _vp)]


class smc_out(C.Structure):
    _fields_ = [("n_loci", C.c_int64), ("loc", _vp), ("cnt", _vp), ("pi", _vp), ("max_allele", _vp), ("second_allele", _vp),
                ("alt_allele", _vp), ("alt_pi", _vp), ("second_pi", _vp), ("fl1", _vp), ("fl2", _vp), ("biallelic", _vp),
                ("fisher_p", _vp), ("fisher_or", _vp), ("dyn_capacity", C.c_int64), ("n_dyn", C.c_int64), ("dyn_locus", _vp),
                ("dyn_kind", _vp), ("dyn_site", _vp), ("dyn_len", _vp), ("dyn_rep_read", _vp), ("dyn_rep_qpos", _vp),
                ("dyn_iskey", _vp), ("dyn_cnt", _vp), ("dyn_pi", _vp), ("dyn_first", _vp)]


class smc_timings(C.Structure):
    _fields_ = [("ms_h2d", C.c_float), ("ms_prep", C.c_float), ("ms_sort", C.c_float), ("ms_pileup", C.c_float),
                ("ms_stats", C.c_float), ("ms_d2h", C.c_float), ("ms_total_device", C.c_float), ("ms_k_pileup", C.c_float),
                ("n_reads", C.c_int64), ("n_loci", C.c_int64), ("n_tile_events", C.c_int64), ("n_pileup_events", C.c_int64),
                ("n_umi_groups", C.c_int64), ("n_dyn", C.c_int64), ("n_fisher", C.c_int64), ("bytes_h2d", C.c_int64),
                ("bytes_d2h", C.c_int64), ("kernel_launches", C.c_int32), ("ms_k_gather", C.c_float), ("ms_k_merge", C.c_float), ("code_mult", C.c_int32),
                ("dyn_capacity", C.c_int32), ("pipe_chunks", C.c_int32), ("pipe_launches", C.c_int32),
                ("ms_read_sort", C.c_float), ("ms_k_read_prep", C.c_float), ("ms_event_sort", C.c_float), ("read_sort_passes", C.c_int32),
                ("read_prep_bytes", C.c_int64)]


class smc_hp_batch(C.Structure):
    _fields_ = [("n", C.c_int64), ("hpLen", C.c_int32), ("bases", _vp), ("n_bases", C.c_int64), ("win_off", _vp), ("win_len", _vp),
                ("win_pos", _vp), ("ref_off", _vp), ("ref_len", _vp), ("alt_off", _vp), ("alt_len", _vp)]


HP_HOMOPOLYMER, HP_LOWCOMP = 1, 2

EXPORTS = ("smc_version", "smc_ctx_create", "smc_ctx_destroy", "smc_last_error", "smc_call_batch", "smc_upload",
           "smc_run_resident", "smc_download", "smc_get_timings", "smc_list_barcodes", "smc_hp_lowcomp", "smc_fisher_exact", "smc_host_alloc",
           "smc_host_free", "smc_set_downsample", "smc_set_barcode_hashes", "smc_draw_sample", "smc_decode_bam", "smc_decoded_dict_umi",
           "smc_inflate_device")

_lib = None


def load():
    """Load libsmc_b200.so (built in-tree by ``__graft_entry__.build()`` / ``python -m smcounter_b200.build``)."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("SMC_B200_LIB", LIB_PATH)      # A/B builds of the same ABI (tuning only)
    if not os.path.exists(path):
        raise ImportError("libsmc_b200.so is not built (%s); run `python -m smcounter_b200.build`. "
                          "smcounter_b200 has no CPU fallback." % LIB_PATH)
    lib = C.CDLL(path)
    lib.smc_version.restype = C.c_int
    lib.smc_ctx_create.argtypes = [C.c_int, C.POINTER(smc_params), C.POINTER(_vp)]
    lib.smc_ctx_create.restype = C.c_int
    lib.smc_ctx_destroy.argtypes = [_vp]
    lib.smc_ctx_destroy.restype = None
    lib.smc_last_error.argtypes = [_vp]
    lib.smc_last_error.restype = C.c_char_p
    lib.smc_call_batch.argtypes = [_vp, C.POINTER(smc_reads_soa), C.POINTER(smc_loci), C.POINTER(smc_umi_keep), C.POINTER(smc_out)]
    lib.smc_call_batch.restype = C.c_int
    lib.smc_upload.argtypes = [_vp, C.POINTER(smc_reads_soa), C.POINTER(smc_loci), C.POINTER(smc_umi_keep)]
    lib.smc_upload.restype = C.c_int
    lib.smc_run_resident.argtypes = [_vp]
    lib.smc_run_resident.restype = C.c_int
    lib.smc_download.argtypes = [_vp, C.POINTER(smc_out)]
    lib.smc_download.restype = C.c_int
    lib.smc_fisher_exact.argtypes = [_vp, C.c_int64, _vp, _vp, _vp]
    lib.smc_fisher_exact.restype = C.c_int
    lib.smc_host_alloc.argtypes = [C.c_int64, C.POINTER(C.c_void_p)]
    lib.smc_host_alloc.restype = C.c_int
    lib.smc_host_free.argtypes = [C.c_void_p]
    lib.smc_host_free.restype = None
    lib.smc_get_timings.argtypes = [_vp, C.POINTER(smc_timings)]
    lib.smc_get_timings.restype = C.c_int
    lib.smc_list_barcodes.argtypes = [_vp, C.c_int64, _vp, _vp, _vp, _vp, C.c_int64]
    lib.smc_list_barcodes.restype = C.c_int
    lib.smc_hp_lowcomp.argtypes = [_vp, C.POINTER(smc_hp_batch), _vp]
    lib.smc_hp_lowcomp.restype = C.c_int
    lib.smc_set_downsample.argtypes = [_vp, C.c_int]
    lib.smc_set_downsample.restype = C.c_int
    lib.smc_set_barcode_hashes.argtypes = [_vp, C.c_int64, _vp, _vp]
    lib.smc_set_barcode_hashes.restype = C.c_int
    lib.smc_draw_sample.argtypes = [_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp]
    lib.smc_draw_sample.restype = C.c_int
    lib.smc_decode_bam.argtypes = [_vp, _vp, C.c_int64, _vp, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_int64, _vp, _vp, _vp, C.c_int32, _vp]
    lib.smc_decode_bam.restype = C.c_int
    lib.smc_decoded_dict_umi.argtypes = [_vp, C.c_int64]
    lib.smc_decoded_dict_umi.restype = C.c_char_p
    lib.smc_inflate_device.argtypes = [_vp, C.c_int64, _vp, C.c_int64, _vp, _vp, _vp, C.c_int64, _vp, _vp, _vp]
    lib.smc_inflate_device.restype = C.c_int
    _lib = lib
    return lib


def ptr(a: np.ndarray | None):
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data
