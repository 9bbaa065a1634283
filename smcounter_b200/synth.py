"""Seeded synthetic UMI-tagged amplicon reads (QIAseq-like), produced directly as ReadsSoA buffers.

Used by tests, ``__graft_entry__.smoke()`` and ``bench.py`` (there is no network for real datasets, and the
reference's example.bam is not distributed).  Shapes follow SURVEY.md section 8(d): paired 2 x ``read_len``
reads, R2 starting at a gene-specific primer and R1 at the random (barcode) end of the fragment, all PCR
copies of one barcode sharing the fragment ends, base qualities 85 % Q37 / 10 % Q30 / 5 % Q12, substitution
errors at 10^(-Q/10), SNV / insertion / deletion sites carried per molecule at a given allele fraction,
occasional soft clips, low-MAPQ reads and per-fragment PCR errors.

Never emitted (the reference's behaviour there is pysam-version dependent, SURVEY.md Appendix A.2): reads that
are neither read1 nor read2, unmapped/secondary flags, N/P CIGAR ops, D adjacent to I, missing qualities.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from .fasta import SparseRef
from .soa import ReadsSoA

_ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
_NIB = np.array([1, 2, 4, 8], dtype=np.uint8)          # BAM nibble of A, C, G, T


@dataclass
class SynthSpec:
    umis_per_locus: float = 300.0     # mean barcodes covering a locus
    rpb: float = 4.0                  # mean fragments (read pairs) per barcode
    read_len: int = 150
    spacing: int = 150                # distance between amplicon anchors
    frag_extra: int = 110             # fragment length is uniform in [read_len, read_len + frag_extra]
    snv_every: int = 1000             # one SNV site per this many target bases (0 = none)
    snv_vaf: float = 0.01
    indel_every: int = 0              # one insertion site and one deletion site per this many bases (0 = none)
    indel_vaf: float = 0.05
    softclip_frac: float = 0.05
    lowmapq_frac: float = 0.02
    pcr_err_per_frag: float = 0.003
    n_frac: float = 0.0005            # fraction of bases called 'N' (quality 2)
    q_values: tuple = (37, 30, 12)
    q_probs: tuple = (0.85, 0.10, 0.05)
    depth_sigma: float = 0.0          # log-normal sigma of per-interval depth (config 5)


def _ref_windows(intervals, chroms, lengths, rng, margin):
    """Random reference bases over each target interval +- margin; returns SparseRef."""
    ref = SparseRef(lengths)
    by_chrom = {}
    for (c, s, e) in intervals:
        by_chrom.setdefault(c, []).append((max(0, s - margin), min(lengths[c], e + margin)))
    for c, spans in by_chrom.items():
        spans.sort()
        merged = []
        for (s, e) in spans:
            if merged and s <= merged[-1][1]:
                merged[-1][1] = max(merged[-1][1], e)
            else:
                merged.append([s, e])
        for (s, e) in merged:
            ref.add_window(c, s, _ACGT[rng.integers(0, 4, size=e - s)])
    return ref


def make_panel(intervals, spec: SynthSpec | None = None, seed: int = 1, chroms=None, lengths=None, umi_base: int = 0):
    """Generate reads for target ``intervals`` = [(chrom, start, end), ...] (0-based half-open, BED style).

    Returns (ReadsSoA in coordinate order, SparseRef, truth dict).
    """
    spec = spec or SynthSpec()
    rng = np.random.Generator(np.random.Philox(seed))
    if chroms is None:
        chroms = []
        for (c, _, _) in intervals:
            if c not in chroms:
                chroms.append(c)
    cidx = {c: i for i, c in enumerate(chroms)}
    rl = spec.read_len
    maxfrag = rl + spec.frag_extra
    margin = maxfrag + 64
    if lengths is None:
        lengths = {c: 0 for c in chroms}
        for (c, s, e) in intervals:
            lengths[c] = max(lengths[c], e + 2 * margin)
    ref = _ref_windows(intervals, chroms, lengths, rng, margin + 64)

    cov_factor = 1.0 + 0.5 * spec.frag_extra / spec.spacing          # barcodes seen per locus / per amplicon
    U_mean = spec.umis_per_locus / cov_factor

    # quality model as lookup tables: a uint8 draw -> quality class, class -> phred / error threshold (of 65536)
    q_lut = np.zeros(256, dtype=np.uint8)
    edges = np.round(np.cumsum(spec.q_probs) * 256).astype(int)
    lo_ = 0
    for qi, hi_ in enumerate(edges):
        q_lut[lo_:hi_] = qi
        lo_ = hi_
    q_lut[lo_:] = len(spec.q_values) - 1
    q_vals8 = np.asarray(spec.q_values, dtype=np.uint8)
    err_thr = np.round(np.power(10.0, -np.asarray(spec.q_values, dtype=np.float64) / 10.0) * 65536).astype(np.uint16)

    cols = {k: [] for k in ("ref_id", "pos", "flag", "mapq", "nm", "umi", "frag", "kind", "k", "ilen")}
    seq_rows, qual_rows = [], []
    truth = {"snv": [], "ins": [], "del": []}
    umi_counter = int(umi_base)
    frag_counter = 0

    for (c, s, e) in intervals:
        depth_scale = float(np.exp(rng.normal(0.0, spec.depth_sigma))) if spec.depth_sigma > 0 else 1.0
        n_amp = max(1, -(-(e - s + 25) // spec.spacing))
        w0 = max(0, s - margin)
        w1 = min(lengths[c], e + margin)
        refarr = ref.fetch_array(c, w0, w1)
        refcode = np.searchsorted(_ACGT, refarr).astype(np.int64) % 4          # A0 C1 G2 T3 (N -> 0)
        refcode8 = refcode.astype(np.uint8)
        swv = np.lib.stride_tricks.sliding_window_view(refcode8, rl)
        # variant sites of this interval (absolute 0-based positions)
        snv_sites = np.array([p for p in range(s, e) if spec.snv_every and p % spec.snv_every == 17 % spec.snv_every],
                             dtype=np.int64)
        ins_sites = np.array([p for p in range(s, e) if spec.indel_every and p % spec.indel_every == 5 % spec.indel_every],
                             dtype=np.int64)
        del_sites = np.array([p for p in range(s, e) if spec.indel_every and
                              p % spec.indel_every == (5 + spec.indel_every // 2) % spec.indel_every], dtype=np.int64)
        for p in snv_sites:
            truth["snv"].append((c, int(p), "ACGT"[(refcode[p - w0] + 1) % 4]))
        for p in ins_sites:
            truth["ins"].append((c, int(p), 1 + int(p) % 3))
        for p in del_sites:
            truth["del"].append((c, int(p), 1 + int(p) % 4))

        for a in range(n_amp):
            fwd_primer = (a % 2 == 0)
            anchor = s - 25 + a * spec.spacing
            if anchor < 0:
                anchor = 0
            nU = int(rng.poisson(U_mean * depth_scale))
            if nU == 0:
                continue
            fraglen = rng.integers(rl, maxfrag + 1, size=nU)
            nfr = 1 + rng.poisson(max(spec.rpb - 1.0, 0.0), size=nU)
            if fwd_primer:
                fs = np.full(nU, anchor, dtype=np.int64)               # fragment start (primer end)
                fe = fs + fraglen
            else:
                fe = np.full(nU, anchor + maxfrag, dtype=np.int64)
                fs = fe - fraglen
            umi = (np.uint64(1) << np.uint64(32)) | (
                (np.arange(umi_counter, umi_counter + nU, dtype=np.uint64) * np.uint64(2654435761)) & np.uint64(0xFFFFFFFF))
            umi_counter += nU
            # per-molecule variants
            mol_snv = rng.random((nU, len(snv_sites))) < spec.snv_vaf if len(snv_sites) else np.zeros((nU, 0), bool)
            mol_indel = np.full(nU, -1, dtype=np.int64)                # index into all_indels or -1
            all_indels = [(int(p), +(1 + int(p) % 3)) for p in ins_sites] + [(int(p), -(1 + int(p) % 4)) for p in del_sites]
            if all_indels:
                pick = rng.random(nU) < spec.indel_vaf * len(all_indels)
                mol_indel[pick] = rng.integers(0, len(all_indels), size=int(pick.sum()))
            # expand to fragments (PCR copies)
            F = int(nfr.sum())
            f_umi = np.repeat(np.arange(nU), nfr)
            f_id = np.arange(frag_counter, frag_counter + F, dtype=np.int64)
            frag_counter += F
            pcr_has = rng.random(F) < spec.pcr_err_per_frag
            pcr_pos = fs[f_umi] + rng.integers(0, rl, size=F)
            pcr_base = rng.integers(0, 4, size=F)
            # two reads per fragment: R2 at the primer end, R1 at the barcode end
            ia = np.array(all_indels, dtype=np.int64).reshape(-1, 2)
            for which in ("R2", "R1"):
                at_start = (which == "R2") == fwd_primer                # read anchored at fragment start?
                reverse = not at_start
                r_fs = fs[f_umi]
                r_fe = fe[f_umi]
                ind = mol_indel[f_umi]
                kind = np.zeros(F, dtype=np.int8)                       # 0 plain, 1 ins, 2 del
                ilen = np.zeros(F, dtype=np.int64)
                vpos = np.zeros(F, dtype=np.int64)
                if len(ia):
                    has = ind >= 0
                    vpos[has] = ia[ind[has], 0]
                    ilen[has] = np.abs(ia[ind[has], 1])
                    kind[has] = np.where(ia[ind[has], 1] > 0, 1, 2)
                # reference span of the read and its start
                span = np.where(kind == 1, rl - ilen, np.where(kind == 2, rl + ilen, rl))
                start = np.where(at_start, r_fs, r_fe - span)
                kk = vpos - start + 1                                   # matched bases before the indel
                ok = (kind > 0) & (kk >= 5) & (np.where(kind == 1, kk + ilen, kk) <= rl - 5)
                kind = np.where(ok, kind, 0).astype(np.int8)
                ilen = np.where(ok, ilen, 0)
                kk = np.where(ok, kk, 0)
                span = np.where(kind == 1, rl - ilen, np.where(kind == 2, rl + ilen, rl))
                start = np.where(at_start, r_fs, r_fe - span)
                neg = start < 0
                if neg.any():                                           # cannot happen for sane BEDs; keep plain
                    start = np.where(neg, 0, start)
                    kind = np.where(neg, 0, kind).astype(np.int8)
                    ilen = np.where(neg, 0, ilen)
                    kk = np.where(neg, 0, kk)

                def col_of(p):
                    """query column of reference position p (array per read) or -1"""
                    d = p - start
                    c = np.where(kind == 2, np.where(d < kk, d, np.where(d >= kk + ilen, d - ilen, -1)),
                                 np.where(kind == 1, np.where(d < kk, d, d + ilen), d))
                    return np.where((d >= 0) & (c >= 0) & (c < rl), c, -1)

                # dense: reference bases as if every read were plain, then fix the rows with an indel
                base = swv[np.clip(start - w0, 0, len(refcode8) - rl)].copy()          # (F, rl) uint8 codes 0..3
                rows_i = np.flatnonzero(kind > 0)
                inserted_cells = None
                if len(rows_i):
                    j = np.arange(rl, dtype=np.int64)[None, :]
                    k_ = kk[rows_i, None]
                    il = ilen[rows_i, None]
                    kd = kind[rows_i, None]
                    refidx = start[rows_i, None] + j
                    refidx = np.where((kd == 2) & (j >= k_), refidx + il, refidx)
                    refidx = np.where((kd == 1) & (j >= k_ + il), refidx - il, refidx)
                    ins_m = (kd == 1) & (j >= k_) & (j < k_ + il)
                    sub = refcode8[np.clip(refidx - w0, 0, len(refcode8) - 1)]
                    sub = np.where(ins_m, ((vpos[rows_i, None] + (j - k_)) % 4).astype(np.uint8), sub)
                    base[rows_i] = sub
                    inserted_cells = (rows_i, ins_m)
                truebase = base.copy()
                if inserted_cells is not None:                                  # inserted bases never count as mismatches
                    pass
                # molecule SNVs (sparse edits)
                for si, p in enumerate(snv_sites):
                    carr = np.flatnonzero(mol_snv[f_umi, si])
                    if len(carr):
                        cc = col_of(np.full(F, p, dtype=np.int64))[carr]
                        m = cc >= 0
                        base[carr[m], cc[m]] = (refcode8[p - w0] + 1) % 4
                # PCR error shared by both reads of the fragment
                rows_p = np.flatnonzero(pcr_has)
                if len(rows_p):
                    cc = col_of(pcr_pos)[rows_p]
                    m = cc >= 0
                    base[rows_p[m], cc[m]] = pcr_base[rows_p[m]].astype(np.uint8)
                # qualities and sequencing errors (dense uint8 / uint16 passes)
                qsel = q_lut[rng.integers(0, 256, size=(F, rl), dtype=np.uint8)]
                qual = q_vals8[qsel]
                err = rng.integers(0, 65536, size=(F, rl), dtype=np.uint16) < err_thr[qsel]
                er, ec = np.nonzero(err)
                if len(er):
                    base[er, ec] = (base[er, ec] + rng.integers(1, 4, size=len(er), dtype=np.uint8)) % 4
                nib = _NIB[base]
                nN = rng.binomial(F * rl, spec.n_frac) if spec.n_frac > 0 else 0
                if nN:
                    nr = rng.integers(0, F, size=nN)
                    nc = rng.integers(0, rl, size=nN)
                    nib[nr, nc] = 15
                    qual[nr, nc] = 2
                # soft clips on plain reads only
                sc = (kind == 0) & (rng.random(F) < spec.softclip_frac)
                sclen = np.where(sc, rng.integers(1, 9, size=F), 0)
                sc_left = sc & (rng.random(F) < 0.5)
                sc_right = sc & ~sc_left
                lclip = np.where(sc_left, sclen, 0)
                rclip = np.where(sc_right, sclen, 0)
                mismatch_cells = nib != _NIB[truebase]
                if inserted_cells is not None:
                    sub = mismatch_cells[inserted_cells[0]]
                    sub[inserted_cells[1]] = False
                    mismatch_cells[inserted_cells[0]] = sub
                rows_c = np.flatnonzero(sc)
                if len(rows_c):
                    j = np.arange(rl, dtype=np.int64)[None, :]
                    clipped = (j < lclip[rows_c, None]) | (j >= rl - rclip[rows_c, None])
                    sub = nib[rows_c]
                    sub[clipped] = _NIB[rng.integers(0, 4, size=int(clipped.sum()))]
                    nib[rows_c] = sub
                    subm = mismatch_cells[rows_c]
                    subm[clipped] = False
                    mismatch_cells[rows_c] = subm
                # NM = mismatches of aligned, non-inserted bases vs the reference + indel length
                nm = mismatch_cells.sum(axis=1) + ilen
                pos = start + lclip
                flag = np.full(F, 0x1 | 0x2, dtype=np.uint16)
                flag |= np.uint16(0x40 if which == "R1" else 0x80)
                flag |= np.uint16(0x10 if reverse else 0x20)
                mapq = np.where(rng.random(F) < spec.lowmapq_frac, 20, 60).astype(np.uint8)
                # kind code for the cigar builder: 0 plain, 1 ins, 2 del, 3 left clip, 4 right clip
                kc = kind.astype(np.int64)
                kc = np.where(sc_left, 3, np.where(sc_right, 4, kc))
                cols["ref_id"].append(np.full(F, cidx[c], dtype=np.int32))
                cols["pos"].append(pos.astype(np.int32))
                cols["flag"].append(flag)
                cols["mapq"].append(mapq)
                cols["nm"].append(nm.astype(np.int32))
                cols["umi"].append(umi[f_umi])
                cols["frag"].append(f_id)
                cols["kind"].append(kc)
                cols["k"].append(np.where(kc == 3, lclip, np.where(kc == 4, rclip, kk)))
                cols["ilen"].append(ilen)
                seq_rows.append(nib)
                qual_rows.append(qual)

    cat = {k: (np.concatenate(v) if v else np.zeros(0, dtype=np.int64)) for k, v in cols.items()}
    n = len(cat["pos"])
    nibs = np.concatenate(seq_rows) if seq_rows else np.zeros((0, rl), np.uint8)
    quals = np.concatenate(qual_rows) if qual_rows else np.zeros((0, rl), np.uint8)
    order = np.lexsort((np.arange(n), cat["pos"], cat["ref_id"]))      # coordinate order, stable
    for k in cat:
        cat[k] = cat[k][order]
    nibs = nibs[order]
    quals = quals[order]
    frag_id = relabel_frag_ids(cat["frag"])
    # cigars
    kc, kk, il = cat["kind"], cat["k"], cat["ilen"]
    n_cigar = np.where(kc == 0, 1, np.where(kc >= 3, 2, 3)).astype(np.uint16)
    cigar_off = np.concatenate(([0], np.cumsum(n_cigar.astype(np.int64))))[:-1]
    cigar = np.zeros(int(n_cigar.sum()), dtype=np.uint32)
    M, I, D, S = 0, 1, 2, 4
    w = lambda length, op: ((length.astype(np.uint32) << np.uint32(4)) | np.uint32(op))
    m = kc == 0
    cigar[cigar_off[m]] = (rl << 4) | M
    m = kc == 1
    cigar[cigar_off[m]] = w(kk[m], M); cigar[cigar_off[m] + 1] = w(il[m], I); cigar[cigar_off[m] + 2] = w(rl - kk[m] - il[m], M)
    m = kc == 2
    cigar[cigar_off[m]] = w(kk[m], M); cigar[cigar_off[m] + 1] = w(il[m], D); cigar[cigar_off[m] + 2] = w(rl - kk[m], M)
    m = kc == 3
    cigar[cigar_off[m]] = w(kk[m], S); cigar[cigar_off[m] + 1] = w(rl - kk[m], M)
    m = kc == 4
    cigar[cigar_off[m]] = w(rl - kk[m], M); cigar[cigar_off[m] + 1] = w(kk[m], S)
    # pack bases
    if rl & 1:
        nibs = np.concatenate((nibs, np.zeros((n, 1), np.uint8)), axis=1)
    packed = ((nibs[:, 0::2] << 4) | nibs[:, 1::2]).astype(np.uint8)
    sb = packed.shape[1] if n else (rl + 1) // 2
    soa = ReadsSoA(
        ref_id=cat["ref_id"].astype(np.int32), pos=cat["pos"].astype(np.int32), flag=cat["flag"].astype(np.uint16),
        mapq=cat["mapq"].astype(np.uint8), nm=cat["nm"].astype(np.int32), l_seq=np.full(n, rl, dtype=np.int32),
        seq_off=np.arange(n, dtype=np.int64) * sb, qual_off=np.arange(n, dtype=np.int64) * rl,
        cigar_off=cigar_off.astype(np.int64), n_cigar=n_cigar, umi=cat["umi"].astype(np.uint64), frag_id=frag_id,
        seq=np.ascontiguousarray(packed).reshape(-1), qual=np.ascontiguousarray(quals).reshape(-1), cigar=cigar,
        chroms=list(chroms))
    return soa, ref, truth


def relabel_frag_ids(frag: np.ndarray) -> np.ndarray:
    """Dense fragment ids in order of first appearance (the canonical fragment order of the C-ABI)."""
    uniq, first, inv = np.unique(frag, return_index=True, return_inverse=True)
    rank = np.empty(len(uniq), dtype=np.int64)
    rank[np.argsort(first, kind="stable")] = np.arange(len(uniq))
    return rank[inv].astype(np.uint32)


def merge_soas(parts, chroms):
    """Concatenate ReadsSoA batches generated for disjoint interval groups and restore coordinate order."""
    parts = [p for p in parts if p.n]
    if not parts:
        raise ValueError("no reads")
    cat = lambda name: np.concatenate([getattr(p, name) for p in parts])
    frag_off = np.cumsum([0] + [int(p.frag_id.max()) + 1 for p in parts])[:-1]
    frag = np.concatenate([p.frag_id.astype(np.int64) + o for p, o in zip(parts, frag_off)])
    seq_off = np.concatenate([p.seq_off + o for p, o in zip(parts, np.cumsum([0] + [p.seq.nbytes for p in parts])[:-1])])
    qual_off = np.concatenate([p.qual_off + o for p, o in zip(parts, np.cumsum([0] + [p.qual.nbytes for p in parts])[:-1])])
    cig_off = np.concatenate([p.cigar_off + o for p, o in zip(parts, np.cumsum([0] + [len(p.cigar) for p in parts])[:-1])])
    ref_id, pos = cat("ref_id"), cat("pos")
    order = np.lexsort((np.arange(len(pos)), pos, ref_id))
    soa = ReadsSoA(ref_id=ref_id[order], pos=pos[order], flag=cat("flag")[order], mapq=cat("mapq")[order], nm=cat("nm")[order],
                   l_seq=cat("l_seq")[order], seq_off=seq_off[order], qual_off=qual_off[order], cigar_off=cig_off[order],
                   n_cigar=cat("n_cigar")[order], umi=cat("umi")[order], frag_id=relabel_frag_ids(frag[order]),
                   seq=cat("seq"), qual=cat("qual"), cigar=cat("cigar"), chroms=list(chroms))
    return soa.repack()          # payload in read order, as a BAM decode delivers it


def _mp_job(args):
    intervals, spec, seed, chroms, lengths, umi_base = args
    return make_panel(intervals, spec, seed=seed, chroms=chroms, lengths=lengths, umi_base=umi_base)


def make_panel_mp(intervals, spec: SynthSpec | None = None, seed: int = 1, workers: int | None = None, n_groups: int | None = None):
    """make_panel() over groups of intervals in worker processes (bench-scale inputs).  Deterministic for a given
    (intervals, spec, seed, number of groups); ``n_groups`` defaults to 4 per worker, so pass it to get the same reads
    whatever the number of workers."""
    import multiprocessing as mp
    import os

    spec = spec or SynthSpec()
    workers = workers or min(16, os.cpu_count() or 1)
    chroms = []
    for (c, _, _) in intervals:
        if c not in chroms:
            chroms.append(c)
    margin = spec.read_len + spec.frag_extra + 64
    lengths = {c: 0 for c in chroms}
    for (c, s, e) in intervals:
        lengths[c] = max(lengths[c], e + 2 * margin)
    ngroups = max(1, min(len(intervals), n_groups or workers * 4))
    groups = [intervals[i::ngroups] for i in range(ngroups)]
    jobs = [(g, spec, seed * 1000003 + i, chroms, lengths, i << 24) for i, g in enumerate(groups)]
    if workers > 1 and ngroups > 1:
        with mp.get_context("fork").Pool(workers) as pool:
            outs = pool.map(_mp_job, jobs)
    else:
        outs = [_mp_job(j) for j in jobs]
    soa = merge_soas([o[0] for o in outs], chroms)
    ref = SparseRef(lengths)
    truth = {"snv": [], "ins": [], "del": []}
    for (_, r, t) in outs:
        for c, ws in r.windows.items():
            for (st, arr) in ws:
                ref.add_window(c, st, arr)
        for k in truth:
            truth[k].extend(t[k])
    return soa, ref, truth


def panel_intervals_from_bed(path, limit=None, seed=None):
    """Read a 3-column BED; optionally take a seeded random subset of ``limit`` intervals (kept in file order)."""
    ivs = []
    with open(path) as fh:
        for line in fh:
            if line.startswith("track ") or not line.strip():
                continue
            c, s, e = line.rstrip("\n").split("\t")[:3]
            ivs.append((c, int(s), int(e)))
    if limit is not None and limit < len(ivs):
        rng = np.random.Generator(np.random.Philox(0 if seed is None else seed))
        keep = np.sort(rng.choice(len(ivs), size=limit, replace=False))
        ivs = [ivs[i] for i in keep]
    return ivs
