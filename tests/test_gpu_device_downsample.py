"""-m gpu: down-sampling drawn on the device (smc_set_downsample(SMC_DS_DEVICE), smc_draw_sample) against
smcounter_b200/downsample.py -- the host draw the product used before, kept as the reference -- and against the oracle's
independent Py2 sampler."""
import numpy as np
import pytest

from helpers import assert_same_results, keep_from_oracle, oracle_run
from py2_sets import code_hash, make_sets, reference_draw
from smcounter_b200 import _ffi
from smcounter_b200.caller import GpuCaller, UmiKeep, VcParams
from smcounter_b200.downsample import draw_keep_masks
from smcounter_b200.rows import device_hp_flags, format_rows
from smcounter_b200.smCounter import _dictionary_hashes, call_loci
from smcounter_b200.synth import SynthSpec, make_panel
from smcounter_b200.targets import build_loci

pytestmark = pytest.mark.gpu

SPEC = SynthSpec(umis_per_locus=50, rpb=3.0, snv_every=30, snv_vaf=0.2, indel_every=45, indel_vaf=0.1)
IVS = [("chr1", 2000, 2050), ("chr2", 400, 420)]


def _mapping(keep):
    return {} if keep is None else {int(l): keep.umi[keep.off[i]:keep.off[i + 1]].tolist() for i, l in enumerate(keep.locus)}


def _rows(caller, res, soa, loci, bed_order, refs, prm):
    hp = device_hp_flags(caller, res, soa, loci, soa.chroms, refs, prm.hpLen)
    return format_rows(res, soa, loci, soa.chroms, refs, prm.hpLen, bed_order, hp_flags=hp)


def host_path(soa, ivs, refs, prm, keep=None):
    """The host draw: call, list the flagged loci's barcodes, draw with downsample.py, call again with every mask."""
    loci, bed_order = build_loci(ivs, soa.chroms, refs)
    c = GpuCaller(prm)
    try:
        res = c.call(soa, loci, keep)
        drawn = draw_keep_masks(c, res, soa, loci, soa.chroms, prm)
        if drawn is not None:
            res = c.call(soa, loci, UmiKeep({**_mapping(keep), **_mapping(drawn)}))
        return _rows(c, res, soa, loci, bed_order, refs, prm), res, _mapping(drawn)
    finally:
        c.close()


def device_path(soa, ivs, refs, prm, keep=None):
    loci, bed_order = build_loci(ivs, soa.chroms, refs)
    c = GpuCaller(prm, device_downsample=True)
    try:
        c.set_barcode_hashes(*_dictionary_hashes(soa.umi, soa.umi_names))
        res = c.call(soa, loci, keep)
        return _rows(c, res, soa, loci, bed_order, refs, prm), res, c.timings()
    finally:
        c.close()


def _same_but_status_bit(a, b):
    """Equal results, except that the device-drawn loci carry SMC_ST_DOWNSAMPLED."""
    sa, sb = a.loc[_ffi.L_STATUS].copy(), b.loc[_ffi.L_STATUS].copy()
    a.loc[_ffi.L_STATUS] &= ~_ffi.ST_DOWNSAMPLED
    b.loc[_ffi.L_STATUS] &= ~_ffi.ST_DOWNSAMPLED
    try:
        assert_same_results(a, b)
    finally:
        a.loc[_ffi.L_STATUS], b.loc[_ffi.L_STATUS] = sa, sb


def _n_flagged(details):
    return sum(1 for d in details if d.get("nBC", 0) > d.get("ds", 1 << 30))


def test_draw_sample_equals_downsample_py():
    sets, names = make_sets(seed=11)
    c = GpuCaller(VcParams(mtDepth=100, rpb=3.0))
    try:
        codes = sorted(names)
        c.set_barcode_hashes(codes, [code_hash(x, names) for x in codes])
        off = np.cumsum([0] + [len(s[0]) for s in sets])
        allc = np.concatenate([np.asarray(s[0], dtype=np.uint64) for s in sets])
        out = c.draw_sample(off, allc, [s[2] for s in sets], [s[3] for s in sets])
        for i, (_, strs, pos1, k) in enumerate(sets):
            assert out[off[i]:off[i] + k].tolist() == reference_draw(strs, pos1, k), (i, len(strs), k, pos1)
        c.set_barcode_hashes([], [])
        top = next(x for x in allc.tolist() if x >> 63)
        with pytest.raises(RuntimeError, match=r"\[-2\].*%016x" % top):
            c.draw_sample([0, 1], [top], [1000], [1])
    finally:
        c.close()


@pytest.mark.parametrize("case", ["low_mtDepth", "maxMT", "trim_compact", "chunks3", "two_shards"])
def test_call_loci_rows_equal_the_oracle_and_the_host_draw(case, monkeypatch):
    prm = VcParams(mtDepth=200, rpb=3.0, maxMT=25) if case == "maxMT" else VcParams(mtDepth=10, rpb=3.0)
    soa, refs, _ = make_panel(IVS, SPEC, seed=23)
    o_rows, details = oracle_run(soa, IVS, refs, prm)
    assert _n_flagged(details) > 20
    h_rows, _, drawn = host_path(soa, IVS, refs, prm)
    assert len(drawn) == _n_flagged(details)
    kw = {}
    if case == "trim_compact":
        soa = soa.trim_to_targets(IVS).compact()
    if case == "chunks3":
        monkeypatch.setenv("SMC_PIPE_CHUNKS", "3")
    if case == "two_shards":
        kw = dict(gpus=2, devices=[0, 0])
    g_rows = call_loci(soa, IVS, refs, prm, **kw)
    assert g_rows == o_rows
    assert g_rows == h_rows
    rows, res, tm = device_path(soa, IVS, refs, prm)
    assert rows == o_rows
    st = res.loc[_ffi.L_STATUS, :res.n_loci]
    assert not (st & _ffi.ST_NEED_DOWNSAMPLE).any()
    assert int(((st & _ffi.ST_DOWNSAMPLED) != 0).sum()) == len(drawn)
    if case == "chunks3":
        assert tm["pipe_chunks"] == 3


@pytest.mark.parametrize("maxMT", [5000, 45000])
def test_one_locus_with_90000_single_read_barcodes(maxMT):
    """random.sample's selection-set branch (maxMT 5000) and its pool branch (45 000) over a dict of 90 000 keys (it grows x2 once beyond 50 000)
    keys: the device mask equals draw_keep_masks' mask, and the device-drawn run equals the host-masked run."""
    from oracle import smcounter_oracle as orc
    from smcounter_b200.soa import records_to_soa
    rng = np.random.default_rng(5)
    ref = "".join(rng.choice(list("ACGT"), size=400))
    refs = orc.DictFasta({"c": ref})
    n = 90000
    bcs = rng.choice(1 << 24, size=n, replace=False)
    recs = [orc.Read("r%d:%s:1" % (i, "".join("ACGT"[(int(b) >> (2 * j)) & 3] for j in range(12))), "c", 90, 0x40 | (0x10 if i % 3 else 0),
                     60, 0, [(0, 40)], ref[90:130], [30] * 40) for i, b in enumerate(bcs)]
    soa = records_to_soa(recs)
    ivs = [("c", 100, 103)]
    prm = VcParams(mtDepth=100, rpb=3.0, maxMT=maxMT)
    _, h_res, drawn = host_path(soa, ivs, refs, prm)
    assert len(drawn) == 3 and all(len(v) == maxMT for v in drawn.values())
    _, d_res, _ = device_path(soa, ivs, refs, prm)
    _same_but_status_bit(d_res, h_res)
    # the device draw through smc_draw_sample on the listed barcodes: the same masks
    loci, _ = build_loci(ivs, soa.chroms, refs)
    c = GpuCaller(prm)
    try:
        res = c.call(soa, loci)
        flagged = np.flatnonzero(res.loc[_ffi.L_STATUS, :loci.n] & _ffi.ST_NEED_DOWNSAMPLE)
        off, umi, first = c.list_barcodes(flagged)
        codes = np.concatenate([umi[off[k]:off[k + 1]][np.argsort(first[off[k]:off[k + 1]], kind="stable")] for k in range(len(flagged))])
        out = c.draw_sample(off, codes, loci.pos0[flagged].astype(np.int64) + 1, [maxMT] * len(flagged))
        for k, i in enumerate(flagged):
            kept = codes[off[k] + out[off[k]:off[k] + maxMT]]
            assert sorted(kept.tolist()) == sorted(drawn[int(i)])
    finally:
        c.close()


def _with_dictionary_barcodes(soa):
    """The same reads with every fourth barcode made unspellable in 2 bits: an N in it, or longer than 31 nt."""
    from oracle import smcounter_oracle as orc
    from smcounter_b200.soa import records_to_soa, soa_to_records
    recs = soa_to_records(soa, orc.Read)
    out, seen = [], {}
    for r in recs:
        rid, bc, x = r.qname.split(":")
        if bc not in seen:
            k = len(seen)
            seen[bc] = bc if k % 4 else (bc[:3] + "N" + bc[4:] if k % 8 else bc * 3)
        out.append(r._replace(qname="%s:%s:%s" % (rid, seen[bc], x)))
    return records_to_soa(out, soa.chroms)


def test_dictionary_coded_barcodes_and_a_missing_hash():
    prm = VcParams(mtDepth=10, rpb=3.0)
    soa0, refs, _ = make_panel(IVS, SPEC, seed=29)
    soa = _with_dictionary_barcodes(soa0)
    assert (soa.umi >> np.uint64(63)).any() and max(len(s) for s in soa.umi_names.values()) > 31
    o_rows, details = oracle_run(soa, IVS, refs, prm)
    assert _n_flagged(details) > 20
    assert call_loci(soa, IVS, refs, prm) == o_rows
    loci, _ = build_loci(IVS, soa.chroms, refs)
    c = GpuCaller(prm, device_downsample=True)
    try:
        with pytest.raises(RuntimeError, match=r"\[-2\] no Py2 hash for the dictionary-coded barcode 0x8"):
            c.call(soa, loci)
    finally:
        c.close()


def test_caller_masks_and_device_draws_in_one_batch():
    prm = VcParams(mtDepth=10, rpb=3.0)
    soa, refs, _ = make_panel(IVS, SPEC, seed=31)
    o_rows, details = oracle_run(soa, IVS, refs, prm)
    _, bo = build_loci(IVS, soa.chroms, refs)
    full = _mapping(keep_from_oracle(details, bo, soa))
    assert len(full) > 20
    part = UmiKeep({l: v for l, v in full.items() if l % 2 == 0})
    h_rows, h_res, drawn = host_path(soa, IVS, refs, prm, part)
    assert drawn and not set(drawn) & set(part.locus.tolist())
    d_rows, d_res, _ = device_path(soa, IVS, refs, prm, part)
    assert d_rows == h_rows == o_rows
    _same_but_status_bit(d_res, h_res)
    st = d_res.loc[_ffi.L_STATUS, :d_res.n_loci]
    assert sorted(np.flatnonzero(st & _ffi.ST_DOWNSAMPLED).tolist()) == sorted(drawn)


def test_mtdepth_zero_leaves_every_covered_locus_without_barcodes():
    prm = VcParams(mtDepth=0, rpb=3.0)
    soa, refs, _ = make_panel(IVS, SPEC, seed=37)
    h_rows, h_res, drawn = host_path(soa, IVS, refs, prm)
    assert drawn and all(len(v) == 0 for v in drawn.values())
    d_rows, d_res, _ = device_path(soa, IVS, refs, prm)
    assert d_rows == h_rows
    _same_but_status_bit(d_res, h_res)
    assert (d_res.loc[_ffi.L_STATUS, :d_res.n_loci] & _ffi.ST_ZERO_COVERAGE).all()
    assert call_loci(soa, IVS, refs, prm) == h_rows


def test_mode_on_without_flagged_loci_changes_nothing():
    prm = VcParams(mtDepth=400, rpb=3.0)
    soa, refs, _ = make_panel(IVS, SPEC, seed=41)
    loci, _ = build_loci(IVS, soa.chroms, refs)
    outs = []
    for on in (False, True):
        c = GpuCaller(prm, device_downsample=on)
        try:
            res = c.call(soa, loci)
            outs.append((res, c.timings()))
        finally:
            c.close()
    (off_res, off_tm), (on_res, on_tm) = outs
    assert not (off_res.loc[_ffi.L_STATUS, :loci.n] & (_ffi.ST_NEED_DOWNSAMPLE | _ffi.ST_DOWNSAMPLED)).any()
    assert_same_results(off_res, on_res)
    assert on_tm["kernel_launches"] == off_tm["kernel_launches"]
