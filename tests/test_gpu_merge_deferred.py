"""-m gpu: barcodes whose calProb takes the general form -- a second allele, a DEL or dynamic allele only, more fragments than
the prior table holds -- are left by k_merge to k_merge_deferred, which replays them from their first fragment code.  These
cases put many such (barcode, locus) pairs into every tile and unit, under keep masks and the device down-sampling, and let the
list of deferred barcodes overflow; every tally, PI and row must still match the oracle."""
import pytest

from helpers import assert_same_results, diff_details, diff_rows, gpu_run, oracle_run, run_case
from smcounter_b200.caller import VcParams
from smcounter_b200.smCounter import call_loci
from smcounter_b200.synth import SynthSpec, make_panel

pytestmark = pytest.mark.gpu

# One PCR error in every fragment (a second allele for a few barcodes at every locus), frequent molecule-level indels (barcodes
# that show a DEL or an insertion only), N bases; six fragments per barcode, so a tile's events span several units.
SPEC = SynthSpec(umis_per_locus=40, rpb=6.0, pcr_err_per_frag=1.0, snv_every=25, snv_vaf=0.2, indel_every=20, indel_vaf=0.3,
                 n_frac=0.002)
IVS = [("chr1", 1000, 1130), ("chr1", 3000, 3070), ("chr2", 500, 600)]
PRM = VcParams(mtDepth=400, rpb=6.0)


def test_deferred_barcodes_over_tiles_units_and_upload_chunks(monkeypatch):
    monkeypatch.setenv("SMC_PIPE_CHUNKS", "4")
    problems, stats, _ = run_case(IVS, SPEC, PRM, seed=101)
    print(stats)
    assert stats["pipe_chunks"] == 4 and stats["pipe_launches"] >= 2
    assert stats["n_dyn"] > 20
    assert not problems, "\n".join(problems)


def test_deferred_barcodes_under_keep_masks():
    """mtDepth 10: ds = 20 barcodes per locus, so nearly every locus is masked to the oracle's draw."""
    problems, stats, _ = run_case(IVS[:2], SPEC, VcParams(mtDepth=10, rpb=6.0), seed=103)
    print(stats)
    assert stats["n_downsampled"] > 100
    assert not problems, "\n".join(problems)


def test_deferred_barcodes_under_device_downsampling():
    """The listing pass of the pileup pair and the second pileup of the device draw, each with its deferred barcodes."""
    prm = VcParams(mtDepth=10, rpb=6.0)
    soa, refs, _ = make_panel(IVS[:2], SPEC, seed=107)
    o_rows, _ = oracle_run(soa, IVS[:2], refs, prm)
    assert call_loci(soa, IVS[:2], refs, prm) == o_rows


def test_deferred_list_overflow_reruns_the_pileup(monkeypatch):
    """A list too short for the batch's deferred barcodes (SMC_SPILL_CAP0: its first length) is noticed after the pileup, which
    runs again (k_gather, k_merge, k_merge_deferred: three more launches) with the list four times longer.  First from length 1,
    which may take several reruns; then from the length that takes exactly one.  The batch defers far fewer barcodes than the
    list's default length (1024), so the first call does not rerun."""
    ivs = [("chr1", 1000, 1030)]
    soa, refs, _ = make_panel(ivs, SPEC, seed=109)
    o_rows, details = oracle_run(soa, ivs, refs, PRM)
    rows0, res0, _, _, tm0 = gpu_run(soa, ivs, refs, PRM)
    assert rows0 == o_rows
    monkeypatch.setenv("SMC_SPILL_CAP0", "1")
    rows1, res1, _, _, tm1 = gpu_run(soa, ivs, refs, PRM)
    reruns = (tm1["kernel_launches"] - tm0["kernel_launches"]) // 3
    assert reruns >= 1 and tm1["kernel_launches"] == tm0["kernel_launches"] + 3 * reruns
    monkeypatch.setenv("SMC_SPILL_CAP0", str(4 ** (reruns - 1)))
    rows2, res2, loci, bed_order, tm2 = gpu_run(soa, ivs, refs, PRM)
    assert tm2["kernel_launches"] == tm0["kernel_launches"] + 3
    for rows, res in ((rows1, res1), (rows2, res2)):
        assert_same_results(res, res0)
        assert rows == o_rows
    problems, _ = diff_details(res2, loci, bed_order, details, soa, refs)
    assert not problems + diff_rows(rows2, o_rows), "\n".join(problems)
