"""Decoders -> columnar tables.  cyvcf2 / pysam (or anything exposing the same API, e.g. the
in-memory fakes the tests install) decode the sites VCF/BCF and the kids' BAM/CRAMs; this module
packs what they yield into the pinned-friendly SoA tables of ``schema.py``.

This is host-side I/O glue (SURVEY 8(f)-2/3: "mate resolution + columnar packer", "streaming site
table"); no phasing arithmetic happens here.
"""
from __future__ import annotations

from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np

from .schema import (AUX_HAS_SA, AUX_SAME_REF, QUAL_ESCAPE, READ_HDR, SITE_FLAG_SIMPLE, ReadTable,
                     SiteTable, pack_seq)


def _merge(intervals: List[Tuple[int, int]]) -> List[Tuple[int, int]]:
    out: List[List[int]] = []
    for a, b in sorted(intervals):
        if out and a <= out[-1][1]:
            out[-1][1] = max(out[-1][1], b)
        else:
            out.append([a, b])
    return [(a, b) for a, b in out]


def pack_sites(vcf, trios: Sequence[Tuple[str, str, str]], regions: Optional[Dict[str, List[Tuple[int, int]]]] = None) -> SiteTable:
    """Trio-major extraction of a joint VCF: the streaming site table of SURVEY 8(f)-3.

    ``vcf``: a cyvcf2.VCF-like handle.  ``regions``: contig -> [(start0, end0)] 0-based half-open
    intervals to decode (None: the whole file).  Every record becomes one row per trio block,
    tagged with the same ``rec_id``.

    One pass over the decoder collects, per record, the four per-sample arrays cyvcf2 hands out
    (gt_types / gt_quals / gt_ref_depths / gt_alt_depths) and five scalars; everything after that --
    the per-trio column gather, the sort by position, the block layout -- is numpy over the stacked
    arrays (no Python work per (record x trio))."""
    samples = list(vcf.samples)
    sidx = {s: i for i, s in enumerate(samples)}
    cols = [(t, [sidx[m] for m in trio]) for t, trio in enumerate(trios) if all(m in sidx for m in trio)]

    def records():
        if regions is None:
            yield from vcf
        else:
            for contig, ivs in regions.items():
                prev_end = None
                for a, b in _merge(ivs):
                    for v in vcf("%s:%d-%d" % (contig, max(a, 0) + 1, max(b, 1))):
                        # a region query returns the records OVERLAPPING it: one that starts before the end of the
                        # previous (disjoint) interval was already returned there.  Two lines of the file that
                        # merely look alike are both kept, as the reference would see both.
                        if prev_end is not None and v.start < prev_end:
                            continue
                        yield v
                    prev_end = max(b, 1)

    chrom: List[str] = []
    pos: List[int] = []
    refs: List[str] = []
    alts_l: List[list] = []
    gts, gqs, rds, ads = [], [], [], []
    for v in records():
        chrom.append(v.CHROM)
        pos.append(v.start)
        refs.append(v.REF)
        alts_l.append(list(v.ALT))
        gts.append(v.gt_types)
        gqs.append(v.gt_quals)
        rds.append(v.gt_ref_depths)
        ads.append(v.gt_alt_depths)
    n = len(pos)
    cindex: Dict[str, int] = {}
    cid = np.fromiter((cindex.setdefault(c, len(cindex)) for c in chrom), dtype=np.int64, count=n)
    simple = np.fromiter((len(al) == 1 and len(r) == 1 and len(al[0]) == 1 and al[0] != "*" for r, al in zip(refs, alts_l)),
                         dtype=bool, count=n)
    ref_b = np.fromiter((ord(r[0]) if r else 0 for r in refs), dtype=np.uint8, count=n)
    alt_b = np.fromiter((ord(al[0][0]) if al and al[0] else 0 for al in alts_l), dtype=np.uint8, count=n)
    ns = len(samples)
    stack = lambda lst, dt: (np.stack([np.asarray(x) for x in lst]).astype(dt, copy=False) if n else np.zeros((0, ns), dtype=dt))
    GT, GQ, RD, AD = stack(gts, np.uint8), stack(gqs, np.float32), stack(rds, np.int32), stack(ads, np.int32)
    refalt = {r: (refs[r], alts_l[r]) for r in np.flatnonzero(~simple).tolist()}
    return build_site_table(trios, cols, list(cindex), cid, np.array(pos, dtype=np.int64), simple, ref_b, alt_b,
                            GT, GQ, RD, AD, refalt)


def build_site_table(trios, cols, contigs: List[str], cid: np.ndarray, pos_a: np.ndarray, simple: np.ndarray,
                     ref_b: np.ndarray, alt_b: np.ndarray, GT: np.ndarray, GQ: np.ndarray, RD: np.ndarray, AD: np.ndarray,
                     refalt: Dict[int, Tuple[str, List[str]]]) -> SiteTable:
    """The trio-major SiteTable of n records in decoder order (``rec_id`` = that order): ``cid`` contig index into
    ``contigs``, ``pos_a`` 0-based start, ``simple`` / ``ref_b`` / ``alt_b`` per record; ``GT`` / ``GQ`` / ``RD`` / ``AD``
    [n, columns] per-sample arrays, ``cols`` [(trio index, [column of kid, dad, mom])] the trios that get blocks;
    ``refalt``: record -> (REF, ALT list) of every record that is not simple."""
    n = int(pos_a.shape[0])
    # block order: (trio, contig id); rows of a block sorted by position, file order among equal positions
    order_in_contig = np.lexsort((np.arange(n), pos_a, cid)) if n else np.zeros(0, dtype=np.int64)
    c_sorted = cid[order_in_contig]
    c_bounds = np.searchsorted(c_sorted, np.arange(len(contigs) + 1))
    keys, offs = [], [0]
    parts = {k: [] for k in ("pos", "flag", "ref", "alt", "gt", "gq", "rd", "ad", "rid")}
    extras: Dict[int, Tuple[str, List[str]]] = {}
    for t, ix in cols:
        ixa = np.array(ix, dtype=np.int64)
        for c in range(len(contigs)):
            rows = order_in_contig[c_bounds[c]: c_bounds[c + 1]]
            if rows.shape[0] == 0:
                continue
            keys.append((t, c))
            parts["pos"].append(pos_a[rows])
            parts["flag"].append(np.where(simple[rows], SITE_FLAG_SIMPLE, 0))
            parts["ref"].append(ref_b[rows])
            parts["alt"].append(alt_b[rows])
            parts["gt"].append(GT[np.ix_(rows, ixa)])
            parts["gq"].append(GQ[np.ix_(rows, ixa)])
            parts["rd"].append(RD[np.ix_(rows, ixa)])
            parts["ad"].append(AD[np.ix_(rows, ixa)])
            parts["rid"].append(rows)
            for local in np.flatnonzero(~simple[rows]).tolist():
                r = int(rows[local])
                extras[offs[-1] + local] = refalt[r]
            offs.append(offs[-1] + rows.shape[0])
    cat = lambda name, dt: (np.concatenate(parts[name]).astype(dt) if parts[name] else np.zeros(0, dtype=dt))
    V = offs[-1]
    tri = lambda name, dt: np.ascontiguousarray(cat(name, dt).reshape(V, 3).T) if V else np.zeros((3, 0), dtype=dt)
    table = SiteTable(
        trios=[tuple(t) for t in trios], contigs=contigs,
        blk_trio=np.array([k[0] for k in keys], dtype=np.int32), blk_contig=np.array([k[1] for k in keys], dtype=np.int32),
        blk_off=np.array(offs, dtype=np.int64), pos=cat("pos", np.int32), flag=cat("flag", np.uint8),
        ref=cat("ref", np.uint8), alt=cat("alt", np.uint8), gt=tri("gt", np.uint8), gq=tri("gq", np.float32),
        rd=tri("rd", np.int32), ad=tri("ad", np.int32), extras=extras, rec_id=cat("rid", np.int64))
    table.validate()
    return table


_BASE_LUT = np.full(256, 1, dtype=np.uint8)          # 2-bit code: any other IUPAC letter -> 1 (escaped)
_ESC_LUT = np.ones(256, dtype=bool)
for _ch, _v in (("A", 0), ("C", 1), ("G", 2), ("T", 3)):
    _BASE_LUT[ord(_ch)] = _v
    _ESC_LUT[ord(_ch)] = False
_BASE_LUT[ord("N")] = 0


def _mate_join(names: List[str], flag: np.ndarray) -> np.ndarray:
    """Index of every read's mate inside one block, or -1: same name, the other segment (0x40 <-> 0x80), a
    primary alignment, the first such read in block order -- what ``bamfile.mate(read)`` resolves to
    (read_collector.py:185,233,400,508) -- for ALL reads with one hashed-name sort instead of one lookup per read."""
    n = len(names)
    mate = np.full(n, -1, dtype=np.int64)
    if n == 0:
        return mate
    h = np.fromiter(map(hash, names), dtype=np.int64, count=n)
    order = np.lexsort((np.arange(n), h))                     # groups of equal hash, block order inside
    hs = h[order]
    first = np.concatenate([[True], hs[1:] != hs[:-1]])
    gid = np.cumsum(first) - 1                                # group of every sorted entry
    G = int(gid[-1]) + 1
    f = flag[order].astype(np.int64)
    primary = (f & 0x900) == 0
    idx_sorted = order
    big = n + 1
    first_r1 = np.full(G, big, dtype=np.int64)
    first_r2 = np.full(G, big, dtype=np.int64)
    np.minimum.at(first_r1, gid[primary & ((f & 0x40) != 0)], idx_sorted[primary & ((f & 0x40) != 0)])
    np.minimum.at(first_r2, gid[primary & ((f & 0x80) != 0)], idx_sorted[primary & ((f & 0x80) != 0)])
    g_of = np.empty(n, dtype=np.int64)
    g_of[order] = gid
    fl = flag.astype(np.int64)
    paired = ((fl & 0x1) != 0) & ((fl & 0x8) == 0)
    cand = np.where((fl & 0x40) != 0, first_r2[g_of], first_r1[g_of])
    ok = paired & (cand < big) & (cand != np.arange(n))
    mate[ok] = cand[ok]
    # a read that is the first candidate of its own group (both segment bits set), a hash collision between two
    # names: resolved one by one (never seen on real data; kept for exactness)
    redo = np.flatnonzero(paired & ((cand == np.arange(n)) | ((cand < big) & ~ok)))
    bad = [i for i in np.flatnonzero(ok).tolist() if names[i] != names[int(mate[i])]] if G < len(set(names)) else []
    if len(redo) or bad:
        by_name: Dict[str, List[int]] = {}
        for i, nm in enumerate(names):
            by_name.setdefault(nm, []).append(i)
        for i in list(redo) + bad:
            i = int(i)
            want = 0x80 if (fl[i] & 0x40) else 0x40
            mate[i] = next((c for c in by_name[names[i]] if c != i and (fl[c] & want) and not (fl[c] & 0x900)), -1)
    return mate


def pack_reads(bams: Dict[str, object], regions: Dict[str, Dict[str, List[Tuple[int, int]]]],
               head_reads: int = 0) -> ReadTable:
    """Reads of every kid overlapping the requested regions, plus their mates, in file order: the mate
    resolution + columnar packer of SURVEY 8(f)-2.

    ``bams``: kid -> pysam.AlignmentFile-like handle.  ``regions``: kid -> contig -> [(start0, end0)].
    ``head_reads``: also keep the template lengths of the first N reads of the file (the reference
    estimates the concordant insert size from the head of the BAM, read_collector.py:11-25);
    they are returned in ``table.head_tlen[kid]``.

    The decoder is walked once per fetched interval; per read only attribute reads remain in Python (one
    list comprehension per column).  CIGAR words, bases, qualities and the mate pointers are built with numpy
    over the whole block: bases through one joined byte string and a 256-entry table, mates through one
    hashed-name sort (``_mate_join``); ``bamfile.mate()`` is only called for the few pairs whose other
    segment lies outside every fetched interval."""
    kids = list(bams)
    contigs: List[str] = []
    cindex: Dict[str, int] = {}
    blocks = []
    head_tlen: Dict[str, np.ndarray] = {}
    for k, kid in enumerate(kids):
        bam = bams[kid]
        if head_reads:
            tl = []
            for i, r in enumerate(bam):
                tl.append(r.tlen)
                if i >= head_reads:
                    break
            head_tlen[kid] = np.array(tl, dtype=np.int64)
        for contig, ivs in regions.get(kid, {}).items():
            rl: List[object] = []
            prev_end = None
            for a, b in _merge(ivs):
                try:
                    it = bam.fetch(contig, max(a, 0), max(b, 1))
                except ValueError:
                    continue
                got = list(it)
                if prev_end is not None:
                    # fetch returns the reads overlapping the interval: one that starts before the end of the
                    # previous (disjoint) interval came back there already
                    got = [r for r in got if r.reference_start >= prev_end or r.reference_end <= prev_end_start]
                rl += got
                prev_end, prev_end_start = max(b, 1), max(a, 0)
            # mates outside the fetched intervals (bamfile.mate(), read_collector.py:185,400): only for the paired
            # primary reads the join leaves without a partner
            names = [r.query_name for r in rl]
            flag = np.fromiter((r.flag for r in rl), dtype=np.int64, count=len(rl))
            mate = _mate_join(names, flag)
            lone = np.flatnonzero((mate < 0) & ((flag & 0x1) != 0) & ((flag & 0x8) == 0) & ((flag & 0x900) == 0))
            seen = {(names[i], int(flag[i]) & 0xC0, rl[i].reference_start) for i in lone.tolist()}
            for i in lone.tolist():
                r = rl[i]
                try:
                    m = bam.mate(r)
                except ValueError:
                    continue
                if getattr(m, "reference_id", 0) != getattr(r, "reference_id", 0):
                    continue
                key = (m.query_name, m.flag & 0xC0, m.reference_start)
                if key in seen:
                    continue
                seen.add(key)
                rl.append(m)
            rl.sort(key=lambda r: r.reference_start)              # stable: file order among equal starts
            if contig not in cindex:
                cindex[contig] = len(contigs)
                contigs.append(contig)
            blocks.append((k, cindex[contig], rl))
    n = sum(len(b[2]) for b in blocks)
    hdr = np.zeros(n, dtype=READ_HDR)
    names_all: List[str] = []
    cig_parts, qual_parts, code_parts = [], [], []
    offs = [0]
    qoff = 0
    coff = 0
    i0 = 0
    for k, c, rl in blocks:
        m = len(rl)
        sl = slice(i0, i0 + m)
        names = [r.query_name for r in rl]
        flag = np.fromiter((r.flag for r in rl), dtype=np.int64, count=m)
        hdr["start"][sl] = np.fromiter((r.reference_start for r in rl), dtype=np.int64, count=m)
        hdr["tlen"][sl] = np.fromiter((r.tlen for r in rl), dtype=np.int64, count=m)
        hdr["flag"][sl] = flag
        hdr["mapq"][sl] = np.fromiter((r.mapping_quality for r in rl), dtype=np.int64, count=m)
        same = np.fromiter((r.next_reference_id == r.reference_id for r in rl), dtype=bool, count=m)
        sa = np.fromiter((r.has_tag("SA") for r in rl), dtype=bool, count=m)
        hdr["aux"][sl] = np.where(same, AUX_SAME_REF, 0) | np.where(sa, AUX_HAS_SA, 0)
        # CIGAR: all (op, length) tuples of the block in one array
        ct = [r.cigartuples or () for r in rl]
        ncig = np.fromiter(map(len, ct), dtype=np.int64, count=m)
        flat = np.array([x for t in ct for x in t], dtype=np.int64).reshape(-1, 2)
        cig_parts.append(((flat[:, 1] << 4) | flat[:, 0]).astype(np.uint32))
        hdr["n_cigar"][sl] = ncig
        hdr["cigar_off"][sl] = coff + np.cumsum(ncig) - ncig
        coff += int(ncig.sum())
        # bases: one joined byte string through the table; qualities: the decoder's byte arrays back to back
        seqs = [r.query_sequence or "" for r in rl]
        lens = np.fromiter(map(len, seqs), dtype=np.int64, count=m)
        b = np.frombuffer("".join(seqs).encode("ascii"), dtype=np.uint8)
        code, esc = _BASE_LUT[b], _ESC_LUT[b]
        qs = [r.query_qualities for r in rl]
        qb = [bytes(q) if (q is not None and len(q) == L) else bytes(int(L)) for q, L in zip(qs, lens.tolist())]
        q = np.frombuffer(b"".join(qb), dtype=np.uint8)
        qual_parts.append(np.where(esc, q | QUAL_ESCAPE, q & 0x7F).astype(np.uint8))
        code_parts.append(code)
        q0 = qoff + np.cumsum(lens) - lens
        hdr["qoff_lo"][sl] = q0 & 0xFFFFFFFF
        hdr["qoff_hi"][sl] = q0 >> 32
        hdr["l_seq"][sl] = lens
        qoff += int(lens.sum())
        mate = _mate_join(names, flag)
        hdr["mate"][sl] = np.where(mate >= 0, mate + i0, -1)
        names_all += names
        i0 += m
        offs.append(i0)
    table = ReadTable(
        kids=kids, contigs=contigs, blk_kid=np.array([b[0] for b in blocks], dtype=np.int32),
        blk_contig=np.array([b[1] for b in blocks], dtype=np.int32), blk_off=np.array(offs, dtype=np.int64),
        hdr=hdr, cigar=np.concatenate(cig_parts).astype(np.uint32) if cig_parts else np.zeros(0, dtype=np.uint32),
        qual=np.concatenate(qual_parts) if qual_parts else np.zeros(0, dtype=np.uint8),
        seq2=pack_seq(np.concatenate(code_parts) if code_parts else np.zeros(0, dtype=np.uint8)), names=names_all)
    table.head_tlen = head_tlen
    table.validate()
    return table
