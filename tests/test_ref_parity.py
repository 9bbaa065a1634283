"""Pins the CPU oracle to the REFERENCE'S OWN CODE (CPU only, no GPU).

``oracle/ref_build.py`` makes /root/reference/smCounter.py executable under Python 3 without touching a line of
calProb / isHPorLowComp / filterVariants / vc (oracle/_ref, git-ignored build output); ``oracle/ref_shims.py`` supplies
the Python-2.7 environment those functions lean on: hash-ordered dict/set models, Py2 round/str, Py2
random.seed/sample, a pysam pileup over the oracle's record model and the four bedtools pipelines of main().

What is asserted here:
  * on the hand-written cases and the whole fuzz corpus (200 seeds, ~20 000 loci) the 45-column row of the reference's
    ``vc()`` equals the oracle's ``vc()`` byte for byte, except for one *classified* kind of difference: an exact PI tie
    between two noise-level alleles that the reference's sequential float sum (in Py2 dict order of the barcodes) breaks
    by one ulp and the oracle's exactly rounded sum keeps (DESIGN.md section 5); at most 1 locus in 5 000 and never with
    PI >= 0.01;
  * ``calProb`` / ``filterVariants`` / ``isHPorLowComp`` called directly on random inputs agree with the oracle's
    restatements (posteriors to 1e-13, flags and FILTER strings identical);
  * the reference's ``main()`` (BED -> loci -> vc -> bedtools repeat filters -> three files) writes the same bytes as the
    oracle's ``run()``;
  * the committed fixture tests/golden/ref_rows.json (made by tests/golden/make_ref_rows.py from the reference's code)
    is what the oracle produces -- this one also runs where /root/reference and oracle/_ref are absent.

The reference is not distributed with this project.  Where it is absent, the vc() comparisons on the cases, the fuzz corpus
and at benchmark depth take the reference's rows from tests/golden/ref_rows.json (every case, the deep cases and the fuzz
seeds stored there); the other comparisons call the reference's functions on fresh inputs and skip.
"""
import functools
import json
import math
import multiprocessing
import os
import random

import pytest

from oracle import ref_build, ref_shims
from oracle import smcounter_oracle as orc
from fuzz import CASES, DEEP_CASES, case_inputs, fuzz_case
from smcounter_b200.soa import soa_to_records
from smcounter_b200.caller import VcParams
from smcounter_b200.synth import SynthSpec, make_panel
from smcounter_b200.targets import loc_list

GOLD = os.path.join(os.path.dirname(__file__), "golden")
needs_ref = pytest.mark.skipif(not ref_build.available(), reason="neither /root/reference nor a prebuilt oracle/_ref is present")

# columns that follow the ALT choice (smCounter.py:541-545, 593): the only ones a PI tie may move
ALT_COLS = {"ALT", "TYPE", "PI", "VDP", "VAF", "VMT", "VMF", "VSM", "FILTER", "REF"}


def _vc_args(prm):
    return (prm.minBQ, prm.minMQ, prm.mtDepth, prm.rpb, prm.hpLen, prm.mismatchThr, prm.mtDrop, prm.maxMT, prm.primerDist)


@functools.lru_cache(maxsize=None)
def stored_ref_rows():
    """{case name: rows} of tests/golden/ref_rows.json: what the reference's vc() printed (Python-2 container order)."""
    with open(os.path.join(GOLD, "ref_rows.json")) as fh:
        return json.load(fh)["cases"]


def both_rows(intervals, spec, prm, seed, order="py2", stored=None):
    """[(oracle row, reference-code row, oracle detail)] for every locus of the case.  The reference's rows come from its own
    vc() where the reference is present, else from case ``stored`` of tests/golden/ref_rows.json."""
    live = ref_build.available()
    assert live or (stored is not None and order == "py2")
    soa, refs, _ = make_panel(intervals, spec, seed=seed)
    index = orc.ReadIndex(soa_to_records(soa, orc.Read))
    if live:
        ref = ref_build.load(order)
        bam = ref_shims.register_bam("mem:%d.bam" % seed, index)
        fa = ref_shims.register_fasta("mem:%d.fa" % seed, refs)
    else:
        want = stored_ref_rows()[stored]
        assert len(want) == len(loc_list(intervals)), stored
    out = []
    for k, (chrom, pos) in enumerate(loc_list(intervals)):
        d = {}
        a = orc.vc(index, chrom, pos, *_vc_args(prm), refs, detail=d)
        b = ref.vc(bam, chrom, pos, *_vc_args(prm), fa) if live else want[k]
        out.append((a, b, d))
    ref_shims.clear_registries()
    return out


def classify(a, b, d):
    """None if the rows are identical, else ('pi_tie', info) for the documented difference, else ('BAD', info)."""
    if a == b:
        return None
    af, bf = a.split("\t"), b.split("\t")
    cols = [orc.headerAll[i] for i in range(45) if af[i] != bf[i]] if len(af) == len(bf) == 45 else ["<shape>"]
    info = (af[0], af[1], [(c, af[orc.headerAll.index(c)], bf[orc.headerAll.index(c)]) for c in cols if c != "<shape>"])
    if not set(cols) <= ALT_COLS or "PI" not in d:
        return ("BAD", info)
    # the reference chose another ALT: legitimate only if that allele's exactly rounded PI ties the oracle's choice
    tied = [k for k, v in d["PI"].items() if abs(v - d["altPI"]) <= 1e-12 * max(v, d["altPI"], 1e-300)]
    if len(tied) >= 2 and d["altPI"] < 0.01:
        return ("pi_tie", info)
    return ("BAD", info)


def _fuzz_worker(seed):
    ivs, spec, prm = fuzz_case(seed)
    n, diffs = 0, []
    for (a, b, d) in both_rows(ivs, spec, prm, seed, stored="fuzz%d" % seed):
        n += 1
        c = classify(a, b, d)
        if c is not None:
            diffs.append((seed,) + c)
    return n, diffs


# ---------------------------------------------------------------------------------------------- recipe
@needs_ref
def test_recipe_leaves_the_hot_path_untouched():
    path = ref_build.build()
    man = json.load(open(ref_build.MANIFEST))
    assert [tuple(e) for e in man["edits"]] == list(ref_build.EDITS) and len(ref_build.EDITS) == 2
    if not os.path.exists(ref_build.REF_SRC):
        pytest.skip("/root/reference absent: prebuilt oracle/_ref in use")
    src = open(ref_build.REF_SRC).read().split("\n")
    gen = open(path).read().split("\n")
    assert len(src) == len(gen)
    changed = [i + 1 for i, (x, y) in enumerate(zip(src, gen)) if x != y]
    assert changed == [e[0] for e in ref_build.EDITS]
    for (lo, hi) in ref_build.HOT_RANGES:
        assert src[lo - 1:hi] == gen[lo - 1:hi]


# ---------------------------------------------------------------------------------------------- vc(): cases + fuzz
@pytest.mark.parametrize("name", sorted(CASES))
def test_reference_vc_equals_oracle_on_cases(name):
    ivs, spec, prm, seed = case_inputs(name)
    rows = both_rows(ivs, spec, prm, seed, stored=name)
    assert len(rows) == sum(e - s for (_, s, e) in ivs)
    bad = [classify(a, b, d) for (a, b, d) in rows if a != b]
    assert not bad, bad[:5]
    if name == "downsample":
        assert sum(1 for (_, _, d) in rows if d.get("nBC", 0) > d.get("ds", 1 << 30)) > 20      # random.sample really ran


FUZZ_SEEDS = list(range(101, 301))


def test_reference_vc_equals_oracle_on_fuzz_corpus():
    if ref_build.available():
        ref_build.load("py2")
        lo, hi = os.environ.get("SMC_REF_FUZZ_SEEDS", "%d:%d" % (FUZZ_SEEDS[0], FUZZ_SEEDS[-1] + 1)).split(":")
        seeds = list(range(int(lo), int(hi)))
    else:
        seeds = sorted(int(k[4:]) for k in stored_ref_rows() if k.startswith("fuzz"))
    ctx = multiprocessing.get_context("fork")
    with ctx.Pool(min(os.cpu_count() or 1, 16)) as pool:
        res = pool.map(_fuzz_worker, seeds, chunksize=1)
    n_loci = sum(n for n, _ in res)
    diffs = [d for _, ds in res for d in ds]
    bad = [d for d in diffs if d[1] == "BAD"]
    ties = [d for d in diffs if d[1] == "pi_tie"]
    print("reference vc() vs oracle vc(): %d seeds, %d loci, %d identical, %d PI-tie differences: %s"
          % (len(seeds), n_loci, n_loci - len(diffs), len(ties), ties))
    assert not bad, bad[:5]
    assert n_loci >= 50 * len(seeds)
    assert len(ties) * 5000 <= n_loci + 5000


@needs_ref
def test_native_order_containers_differ_only_in_tie_breaks():
    """order='native' (plain insertion-ordered dicts; the flavour bench.py times) may differ from order='py2' only where a
    dict order decides something -- the ALT picked among exactly tied PIs (most often A/C/T/G all 0.0 at a clean locus:
    Py2 order says A, C, T, G; insertion order says A, T, G, C).  Every other column must be identical."""
    ivs, spec, prm, seed = case_inputs("snv_basic")
    a = both_rows(ivs, spec, prm, seed, order="py2")
    b = both_rows(ivs, spec, prm, seed, order="native")
    n_diff = 0
    for (x, y) in zip(a, b):
        xf, yf = x[1].split("\t"), y[1].split("\t")
        cols = {orc.headerAll[i] for i in range(45) if xf[i] != yf[i]}
        assert cols <= ALT_COLS, cols
        if cols and "ALT" not in cols:
            # the plain containers iterate in the order of this process's string hashes (PYTHONHASHSEED): the reference's float
            # sum over the barcodes can then land one ulp away and print another last digit of PI -- nothing else may move
            assert cols <= {"PI"}, cols
        elif cols:
            n_diff += 1
            tied = [k for k, v in x[2]["PI"].items() if abs(v - x[2]["altPI"]) <= 1e-12 * max(abs(v), abs(x[2]["altPI"]), 1e-300)]
            assert len(tied) >= 2
    print("rows whose ALT differs between the container flavours:", n_diff, "of", len(a))
    assert n_diff < len(a)            # how many ties fall the other way depends on this process's string hashes (0 .. most)


# ---------------------------------------------------------------------------------------------- calProb
def _random_barcode(rng, py2dict):
    alleles = ["A", "C", "G", "T", "DEL", "N", "INS|A|AT", "DEL|GT|G", "INS|C|CAAG"]
    k = rng.choice([1, 1, 2, 2, 3, 5])
    use = rng.sample(alleles, k)
    n = rng.choice([1, 2, 3, 8, 20])
    frags = []
    for i in range(n):
        base = use[0] if rng.random() < 0.8 else rng.choice(use)
        q = rng.choice([12, 20, 30, 37, 40])
        frags.append([base, 10.0 ** (-q / 10.0), rng.choice(["Paired", "Paired", "R1", "R2"]), i])
    one_bc = py2dict(list)
    for i, f in enumerate(frags):
        one_bc["M0:%d:%d" % (rng.randrange(10 ** 6), i)].append(f[:3])
    return frags, one_bc


@needs_ref
def test_reference_calprob_vs_oracle():
    ref = ref_build.load("py2")
    rng = random.Random(7)
    worst, n_exact, n = 0.0, 0, 0
    for _ in range(3000):
        mtDrop = rng.choice([0, 0, 1, 2])
        frags, one_bc = _random_barcode(rng, ref_shims.Py2DefaultDict)
        want = orc.cal_prob(frags, mtDrop)
        got = ref.calProb(one_bc, mtDrop)
        assert sorted(got.keys()) == sorted(want.keys())
        for k in want:
            n += 1
            a, b = want[k], got[k]
            if a == b:
                n_exact += 1
            else:
                worst = max(worst, abs(a - b) / max(abs(a), abs(b)))
    print("calProb: %d posteriors, %d bit-identical, worst rel err %.2e" % (n, n_exact, worst))
    assert worst < 1e-13          # product order inside a barcode (Py2 dict order of read ids vs first appearance)
    assert n_exact > 0.7 * n


# ---------------------------------------------------------------------------------------------- filterVariants / isHPorLowComp
@needs_ref
def test_reference_is_hp_or_low_comp_vs_oracle():
    ref = ref_build.load("py2")
    rng = random.Random(11)
    seq = "".join(rng.choice("ACGT") for _ in range(200))
    seq = seq[:40] + "A" * 9 + seq[49:90] + "CACACACACACACACACACACA" + seq[112:150] + "GGGGGGGGGGGG" + seq[162:]
    refs = orc.DictFasta({"c": seq})
    fa = ref_shims.register_fasta("mem:hp.fa", refs)
    seen = set()
    for pos in range(1, len(seq) + 1):
        for (refb, altb) in ((seq[pos - 1], "A"), (seq[pos - 1], seq[pos - 1] + "AA"), (seq[pos - 1:pos + 3], seq[pos - 1])):
            for hp in (4, 8, 10):
                want = orc.is_hp_or_low_comp("c", str(pos), hp, refb, altb, refs)
                got = ref.isHPorLowComp("c", str(pos), hp, refb, altb, fa)
                assert tuple(map(bool, got)) == tuple(map(bool, want)), (pos, refb, altb, hp)
                seen.add(tuple(map(bool, got)))
    assert len(seen) == 4
    ref_shims.clear_registries()


@needs_ref
def test_reference_filter_variants_vs_oracle():
    ref = ref_build.load("py2")
    rng = random.Random(13)
    seq = "".join(rng.choice("ACGT") for _ in range(300))
    refs = orc.DictFasta({"c": seq})
    fa = ref_shims.register_fasta("mem:fv.fa", refs)
    DD = ref_shims.Py2DefaultDict
    tags = set()
    for it in range(1500):
        pos = rng.randrange(30, 270)
        origRef = seq[pos - 1]
        origAlt = rng.choice([b for b in "ACGT" if b != origRef] + ["INS|%s|%sAC" % (origRef, origRef)])
        ref_, alt_, vtype = orc.convert_to_vcf(origRef, origAlt)
        big = rng.random() < 0.3

        def cnt(lo, hi):
            return rng.randrange(lo, hi * (40 if big else 1))

        def dd(kind, **kv):
            d = DD(kind)
            for k, v in kv.items():
                d[{"r": origRef, "a": origAlt}[k]] = v
            return d
        usedMT = cnt(1, 60)
        strong = dd(int, a=rng.choice([0, 1, 2, 9]))
        MTCnt = dd(int, a=min(usedMT, cnt(0, 60)), r=cnt(0, 60))
        nalt = cnt(1, 50)
        alleleCnt = dd(int, r=cnt(1, 500), a=nalt)
        cvg = alleleCnt[origRef] + nalt + cnt(0, 10)
        discord = dd(int, a=rng.choice([0, 3, 800, 1500]))
        concord = dd(int, a=rng.choice([0, 5, 700]))
        rev = dd(int, r=cnt(0, 300), a=rng.choice([0, 0, cnt(0, 40)]))
        fwd = dd(int, r=cnt(0, 300), a=rng.choice([0, cnt(0, 40)]))
        lowq = dd(int)
        if rng.random() < 0.5:
            lowq[origAlt] = rng.randrange(0, nalt + 1)

        def ends(nr, na, near_alt):
            return dd(list, r=[rng.randrange(0, 150) for _ in range(nr)],
                      a=[rng.randrange(0, 6) if rng.random() < near_alt else rng.randrange(21, 150) for _ in range(na)])
        r1 = ends(cnt(0, 120), cnt(0, 30), rng.choice([0.0, 0.5, 1.0]))
        r2 = ends(cnt(0, 120), cnt(0, 30), rng.choice([0.0, 0.5, 1.0]))
        r2p = ends(cnt(0, 120), cnt(0, 30), rng.choice([0.0, 0.5, 1.0]))
        primerDist = rng.choice([0, 2, 10])
        hpLen = rng.choice([4, 8, 10])
        args = (usedMT, strong, "c", str(pos), hpLen)
        rest = (MTCnt, alleleCnt, cvg, discord, concord, rev, fwd, lowq, r1, r2, r2p, primerDist)
        want = orc.filter_variants(ref_, alt_, vtype, origAlt, origRef, *args, refs, *rest)
        got = ref.filterVariants(ref_, alt_, vtype, origAlt, origRef, *args, fa, *rest)
        assert got == want, (it, got, want)
        tags.update(t for t in got.split(";") if t)
    print("filterVariants tags seen:", sorted(tags))
    assert {"LM", "LSM", "DP", "SB", "LowQ", "R1CP", "R2CP", "PrimerCP"} <= tags
    ref_shims.clear_registries()


# ---------------------------------------------------------------------------------------------- main()
@needs_ref
def test_reference_main_writes_the_files_the_oracle_writes(tmp_path):
    """The reference's main() end to end (smCounter.py:645-909) -- dict-style args, BED with a track line and overlapping
    intervals, bedtools merge/sort/intersect via the shim, the repeat loop, threshold, the three writers."""
    ref = ref_build.load("py2")
    ivs = [("chr1", 1000, 1150), ("chr2", 600, 640), ("chr1", 1100, 1120)]
    from smcounter_b200.synth import SynthSpec
    spec = SynthSpec(umis_per_locus=80, rpb=3.0, snv_every=40, snv_vaf=0.2, indel_every=60, indel_vaf=0.15)
    soa, refs, _ = make_panel(ivs, spec, seed=31)
    recs = soa_to_records(soa, orc.Read)
    bam = ref_shims.register_bam("mem:main.bam", recs)
    fa = ref_shims.register_fasta("mem:main.fa", refs)
    bed_lines = ["track name=t\n"] + ["%s\t%d\t%d\n" % iv for iv in ivs]
    (tmp_path / "t.bed").write_text("".join(bed_lines))
    trf_rows = [("chr1", "1010", "1040"), ("chr2", "0", "700")]
    rm_rows = [("chr1", "1030", "1060", "Simple_repeat"), ("chr1", "1055", "1100", "Low_complexity"), ("chr1", "1101", "1105", "Satellite"),
               ("chr2", "610", "620", "L1")]
    (tmp_path / "trf.bed").write_text("".join("\t".join(r) + "\n" for r in trf_rows))
    (tmp_path / "rm.bed").write_text("".join("\t".join(r) + "\n" for r in rm_rows))
    prefix = str(tmp_path / "ref")
    ref.parser = None
    thr = ref.main({"outPrefix": prefix, "bamFile": bam, "bedTarget": str(tmp_path / "t.bed"), "mtDepth": 80, "rpb": 3.0, "refGenome": fa,
                    "bedTandemRepeats": str(tmp_path / "trf.bed"), "bedRepeatMaskerSubset": str(tmp_path / "rm.bed"), "bedtoolsPath": "/nowhere/",
                    "threshold": 20})
    want_thr, all_txt, cut_txt, cut_vcf = orc.run(recs, bed_lines, refs, mtDepth=80, rpb=3.0, threshold=20, outPrefix=prefix,
                                                   trf_rows=trf_rows, rm_rows=rm_rows)
    assert thr == want_thr == 20
    assert open(prefix + ".smCounter.all.txt").read() == all_txt
    assert open(prefix + ".smCounter.cut.txt").read() == cut_txt
    assert open(prefix + ".smCounter.cut.vcf").read() == cut_vcf
    assert cut_txt.count("\n") > 3 and "RepT" in all_txt and ("RepS" in all_txt or "LowC" in all_txt)
    assert not [f for f in os.listdir(tmp_path) if ".tmp." in f]                 # :737-740
    ref_shims.clear_registries()


# ---------------------------------------------------------------------------------------------- committed fixture
def test_oracle_reproduces_the_committed_reference_rows():
    """tests/golden/ref_rows.json: rows printed by the REFERENCE'S vc() (tests/golden/make_ref_rows.py, run in the build
    container where /root/reference exists).  The oracle must reproduce every one of them -- no reference needed here."""
    with open(os.path.join(GOLD, "ref_rows.json")) as fh:
        fx = json.load(fh)
    assert fx["source_sha256"] and len(fx["cases"]) >= 8
    n = 0
    for name, want in fx["cases"].items():
        if name.startswith("fuzz"):
            seed = int(name[4:])
            ivs, spec, prm = fuzz_case(seed)
        else:
            ivs, spec, prm, seed = case_inputs(name)
        soa, refs, _ = make_panel(ivs, spec, seed=seed)
        index = orc.ReadIndex(soa_to_records(soa, orc.Read))
        got = [orc.vc(index, chrom, pos, *_vc_args(prm), refs) for (chrom, pos) in loc_list(ivs)]
        assert got == want, name
        n += len(got)
    assert n > 1000


# ---------------------------------------------------------------------------------------------- vc() at the depths of BASELINE.json's configs
DEEP_TASKS = [  # (name, SynthSpec keywords, VcParams keywords, interval, seed)
    ("cfg2", dict(umis_per_locus=3000, rpb=4.0, snv_every=7, snv_vaf=0.01), dict(mtDepth=3000, rpb=4.0), ("chr1", 5000 + 40 * k, 5008 + 40 * k), 900 + k)
    for k in range(4)] + [
    ("cfg1", dict(umis_per_locus=4000, rpb=9.8, snv_every=5, snv_vaf=0.02, indel_every=9, indel_vaf=0.02), dict(mtDepth=3612, rpb=8.6, mtDrop=1, hpLen=8),
     ("chr17", 41243700 + 30 * k, 41243705 + 30 * k), 910 + k) for k in range(2)] + [
    ("cfg3", dict(umis_per_locus=20000, rpb=4.0, snv_every=3, snv_vaf=0.005), dict(mtDepth=20000, rpb=4.0), ("chr2", 7000 + 50 * k, 7002 + 50 * k), 920 + k)
    for k in range(2)]


def _deep_worker(task):
    name, spec_kw, prm_kw, iv, seed, stored = task
    rows = both_rows([iv], SynthSpec(**spec_kw), VcParams(**prm_kw), seed, stored=stored)
    return name, len(rows), [(name, seed) + c for c in (classify(a, b, d) for (a, b, d) in rows) if c is not None], \
        max(d.get("nBC", 0) for (_, _, d) in rows)


def test_reference_vc_equals_oracle_at_benchmark_depth():
    """The same comparison at the depths the BASELINE.json configurations run at (3 000 / 4 000 / 20 000 barcodes per locus,
    rpb 4 / 9.8): thousands of barcodes go through the Python-2 dict models and calProb per locus, PI sums run over thousands
    of terms in dict order on the reference side and exactly here.  Without the reference: the deep cases of fuzz.DEEP_CASES,
    whose reference rows tests/golden/ref_rows.json keeps."""
    if ref_build.available():
        ref_build.load("py2")
        tasks = [t + (None,) for t in DEEP_TASKS]
    else:
        tasks = [(name[len("deep_"):], spec_kw, prm_kw, ivs[0], seed, name) for name, (spec_kw, prm_kw, ivs, seed) in sorted(DEEP_CASES.items())]
    ctx = multiprocessing.get_context("fork")
    with ctx.Pool(min(os.cpu_count() or 1, len(tasks))) as pool:
        res = pool.map(_deep_worker, tasks, chunksize=1)
    n = sum(r[1] for r in res)
    diffs = [d for r in res for d in r[2]]
    print("reference vc() vs oracle at depth: %d loci, deepest %s barcodes, differences: %s" % (n, max(r[3] for r in res), diffs))
    assert n == sum(t[3][2] - t[3][1] for t in tasks)
    assert not [d for d in diffs if d[2] == "BAD"], diffs[:5]
    assert max(r[3] for r in res if r[0] == "cfg3") > 12000 and max(r[3] for r in res if r[0] == "cfg2") > 2000
