"""Columnar (SoA) tables shared by the host packers, the CUDA engine and the oracle.

This file is the single source of truth for the memory layout; ``include/unfazed_sm100.h``
restates it for the C ABI.  Nothing in here touches a GPU.

Layout summary (all little endian, all arrays C-contiguous):

* ``SiteTable`` -- one *block* per (trio, contig), rows sorted by ``pos``.  Trio-major
  extraction of the joint sites VCF: per row ``pos i32``, ``flag u8`` (bit0 = record passes the
  reference's simple-SNV prefilter, informative_site_finder.py:239-244), ``ref/alt u8`` (ASCII
  base, only meaningful when bit0 is set) and three member planes (kid, dad, mom) of
  ``gt u8`` (cyvcf2 codes, utils.py:2-5), ``gq f32``, ``rd i32``, ``ad i32`` -> the 44 B/row
  "canonical layout" of SURVEY.md 8(a)-3.
* ``ReadTable`` -- one block per (kid, contig), reads in BAM file order (sorted by start).
  A 32-byte AoS header per read + three blobs: BAM-encoded CIGAR words, qualities (bit7 of a
  quality byte flags "base is not A/C/G/T": then the 2-bit code is 0 for ``N`` and 1 for any
  other IUPAC letter) and 2-bit packed bases indexed in parallel with the quality blob.
* ``DnmBatch`` -- the de novo variants of one call, with the window plan the host derived from
  ``find``/``find_many`` semantics.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

# genotype codes, cyvcf2 gt_types (reference utils.py:2-5)
HOM_REF, HET, GT_UNKNOWN, HOM_ALT = 0, 1, 2, 3

KID, DAD, MOM = 0, 1, 2

SITE_FLAG_SIMPLE = 1  # len(ALT)==1, len(REF)==1, len(ALT[0])==1, ALT != '*'

# 32-byte read header; mirrored by `struct UnfzRead` in include/unfazed_sm100.h
READ_HDR = np.dtype(
    [
        ("start", "<i4"),      # reference_start, 0-based
        ("tlen", "<i4"),       # template_length
        ("mate", "<i4"),       # global index of the mate record in this table, -1 = mate() raises
        ("cigar_off", "<u4"),  # first CIGAR word
        ("qoff_lo", "<u4"),    # low 32 bits of the base/quality index of query base 0
        ("l_seq", "<i4"),      # query length
        ("flag", "<u2"),       # SAM FLAG
        ("n_cigar", "<u2"),
        ("mapq", "u1"),
        ("aux", "u1"),         # bit0: next_reference_id == reference_id, bit1: has SA tag
        ("qoff_hi", "u1"),     # bits 32..39 of the base/quality index
        ("pad", "u1"),
    ],
    align=False,
)
assert READ_HDR.itemsize == 32

AUX_SAME_REF = 1
AUX_HAS_SA = 2
AUX_HAS_N = 4      # device copies only: some base of the read is not A/C/G/T (set by unfz_expand_nlist)


def min_base_qual(min_gt_qual) -> int:
    """--min-gt-qual as the integer base-quality threshold (read_collector.py:361-362): a phred
    value q is an integer, so ``q < t`` is ``q < ceil(t)``; clamped to the 7 bits a quality has."""
    t = float(min_gt_qual)
    if t <= 0:
        return 0
    if t >= 128:
        return 128
    return int(np.ceil(t))

# BAM CIGAR op codes (pysam cigartuples; reference utils.py:13-24)
CIG_M, CIG_I, CIG_D, CIG_N, CIG_S, CIG_H, CIG_P, CIG_EQ, CIG_X, CIG_B = range(10)

BASE2 = {"A": 0, "C": 1, "G": 2, "T": 3}
BASE_CHARS = "ACGT"
QUAL_ESCAPE = 0x80  # quality byte bit7: base is not one of ACGT


@dataclass
class SiteTable:
    trios: List[Tuple[str, str, str]]          # (kid, dad, mom) sample ids per trio
    contigs: List[str]                         # contig names as spelled in the VCF
    blk_trio: np.ndarray                       # i32[B]
    blk_contig: np.ndarray                     # i32[B]
    blk_off: np.ndarray                        # i64[B+1] row offsets
    pos: np.ndarray                            # i32[V]
    flag: np.ndarray                           # u8[V]
    ref: np.ndarray                            # u8[V]
    alt: np.ndarray                            # u8[V]
    gt: np.ndarray                             # u8[3,V]
    gq: np.ndarray                             # f32[3,V]
    rd: np.ndarray                             # i32[3,V]
    ad: np.ndarray                             # i32[3,V]
    # host-only: full REF / ALT strings of rows that are not simple SNVs
    extras: Dict[int, Tuple[str, List[str]]] = field(default_factory=dict)
    # host-only: identity of the VCF record a row was extracted from.  A joint VCF packed
    # trio-major repeats every record once per trio block; rows sharing a rec_id are ONE record
    # (matters only for get_refalt, snv_phaser.py:73-84).  None = every row is its own record.
    rec_id: Optional[np.ndarray] = None

    @property
    def n_rows(self) -> int:
        return int(self.pos.shape[0])

    def record_ids(self) -> np.ndarray:
        if self.rec_id is None:
            return np.arange(self.n_rows, dtype=np.int64)
        return self.rec_id

    @property
    def n_blocks(self) -> int:
        return int(self.blk_trio.shape[0])

    def block_of(self, trio: int, contig: str) -> int:
        """Block index of (trio, contig name) or -1."""
        key = (trio, contig)
        idx = getattr(self, "_blk_index", None)
        if idx is None:
            idx = {
                (int(t), self.contigs[int(c)]): b
                for b, (t, c) in enumerate(zip(self.blk_trio, self.blk_contig))
            }
            object.__setattr__(self, "_blk_index", idx)
        return idx.get(key, -1)

    def ref_alts(self, row: int) -> Tuple[str, List[str]]:
        """REF string and ALT list of a row, as cyvcf2 would report them."""
        if row in self.extras:
            return self.extras[row]
        return chr(self.ref[row]), [chr(self.alt[row])]

    def validate(self) -> None:
        V = self.n_rows
        assert self.blk_off[0] == 0 and self.blk_off[-1] == V
        for name in ("flag", "ref", "alt"):
            a = getattr(self, name)
            assert a.dtype == np.uint8 and a.shape == (V,), name
        assert self.pos.dtype == np.int32 and self.pos.shape == (V,)
        assert self.gt.dtype == np.uint8 and self.gt.shape == (3, V)
        assert self.gq.dtype == np.float32 and self.gq.shape == (3, V)
        assert self.rd.dtype == np.int32 and self.rd.shape == (3, V)
        assert self.ad.dtype == np.int32 and self.ad.shape == (3, V)
        for b in range(self.n_blocks):
            p = self.pos[self.blk_off[b]: self.blk_off[b + 1]]
            assert np.all(p[1:] >= p[:-1]), "site block %d not sorted" % b


@dataclass
class ReadTable:
    kids: List[str]
    contigs: List[str]                          # contig names as spelled in the BAM
    blk_kid: np.ndarray                         # i32[B]
    blk_contig: np.ndarray                      # i32[B]
    blk_off: np.ndarray                         # i64[B+1] read offsets
    hdr: np.ndarray                             # READ_HDR[N]
    cigar: np.ndarray                           # u32[sum n_cigar], BAM encoding len<<4|op
    qual: np.ndarray                            # u8[Q]
    seq2: np.ndarray                            # u8[ceil(Q/4)], base i at bits 2*(i&3) of byte i>>2
    names: Optional[List[str]] = None           # per read; None -> synthesized from pair id
    # a table whose bases and qualities were decoded on the device only (bamio.read_regions(engine=...)) has
    # qual = seq2 = None and records its number of query bases here
    n_bases: Optional[int] = None

    @property
    def n_reads(self) -> int:
        return int(self.hdr.shape[0])

    @property
    def n_qual(self) -> int:
        """Number of query bases (the length of the quality / base columns)."""
        return int(self.n_bases) if self.qual is None else int(self.qual.shape[0])

    def _need_bases(self, what: str) -> None:
        if self.qual is None:
            raise ValueError("%s needs the quality bytes: this ReadTable was decoded on the device and carries no "
                             "qual / seq2 columns (use its device_reads, or read the file with engine=None)" % what)

    def max_l_seq(self) -> int:
        """Longest read (cached: a pass over the strided header field costs tens of ms at 20 M reads)."""
        m = self.__dict__.get("_max_l_seq")
        if m is None or m[0] != self.hdr.shape[0]:
            m = (self.hdr.shape[0], int(self.hdr["l_seq"].max()) if self.hdr.shape[0] else 0)
            self.__dict__["_max_l_seq"] = m
        return m[1]

    @property
    def n_blocks(self) -> int:
        return int(self.blk_kid.shape[0])

    def block_of(self, kid: int, contig: str) -> int:
        idx = getattr(self, "_blk_index", None)
        if idx is None:
            idx = {
                (int(k), self.contigs[int(c)]): b
                for b, (k, c) in enumerate(zip(self.blk_kid, self.blk_contig))
            }
            object.__setattr__(self, "_blk_index", idx)
        return idx.get((kid, contig), -1)

    def qoff(self, r: int) -> int:
        h = self.hdr[r]
        return int(h["qoff_lo"]) | (int(h["qoff_hi"]) << 32)

    def name_of(self, r: int) -> str:
        if self.names is not None:
            return self.names[r]
        m = int(self.hdr["mate"][r])
        return "q%d" % (min(r, m) if m >= 0 else r)

    def pair_ids(self) -> np.ndarray:
        """Dense per-read id of its pair (the lower index of the two mates): what a synthesized read name is made of.
        Cached; a table packed from a BAM carries ``names`` instead."""
        p = self.__dict__.get("_pair_ids")
        if p is None or p.shape[0] != self.n_reads:
            m = self.hdr["mate"].astype(np.int64)
            r = np.arange(self.n_reads, dtype=np.int64)
            p = np.where(m >= 0, np.minimum(r, m), r)
            self.__dict__["_pair_ids"] = p
        return p

    def names_of(self, idx: np.ndarray) -> List[str]:
        """query_name of many reads at once (both mates of a pair share it)."""
        idx = np.asarray(idx, dtype=np.int64)
        if self.names is not None:
            nm = self.names
            return [nm[i] for i in idx.tolist()]
        return ["q%d" % i for i in self.pair_ids()[idx].tolist()]

    def lowq_plane(self, min_bq: int, chunk: int = 1 << 26) -> np.ndarray:
        """One bit per query base, bit i&7 of byte i>>3: ``(qual & 0x7f) < min_bq``.  This is what the
        device gets instead of the quality bytes -- every base-quality test of the path is this one
        comparison (reference read_collector.py:44-46, :123, :281-284)."""
        self._need_bases("lowq_plane")
        Q = int(self.qual.shape[0])
        out = np.zeros((Q + 7) // 8, dtype=np.uint8)
        for a in range(0, Q, chunk):
            b = min(Q, a + chunk)                          # chunk is a multiple of 8
            out[a >> 3: (b + 7) >> 3] = np.packbits((self.qual[a:b] & 0x7F) < min_bq, bitorder="little")
        return out

    def n_index(self, chunk: int = 1 << 26) -> np.ndarray:
        """Sorted base indices of the non-ACGT bases (quality bit7)."""
        self._need_bases("n_index")
        Q = int(self.qual.shape[0])
        parts = [np.flatnonzero(self.qual[a: a + chunk] & QUAL_ESCAPE) + a for a in range(0, Q, chunk)]
        return np.concatenate(parts).astype(np.int64) if parts else np.zeros(0, dtype=np.int64)

    def ref_ends(self) -> np.ndarray:
        """reference_end (exclusive) of every read: start + lengths of M/D/N/=/X ops. Cached."""
        e = getattr(self, "_ref_ends", None)
        if e is None:
            ops = self.cigar & 15
            ln = (self.cigar >> 4).astype(np.int64)
            consume = np.isin(ops, (CIG_M, CIG_D, CIG_N, CIG_EQ, CIG_X))
            csum = np.concatenate([[0], np.cumsum(np.where(consume, ln, 0))])
            o = self.hdr["cigar_off"].astype(np.int64)
            n = self.hdr["n_cigar"].astype(np.int64)
            e = self.hdr["start"].astype(np.int64) + csum[o + n] - csum[o]
            object.__setattr__(self, "_ref_ends", e)
        return e

    def validate(self) -> None:
        assert self.hdr.dtype == READ_HDR
        assert self.cigar.dtype == np.uint32
        if self.qual is None:
            assert self.seq2 is None and self.n_bases is not None
            assert self.n_bases == int(self.hdr["l_seq"].astype(np.int64).sum())
        else:
            assert self.qual.dtype == np.uint8 and self.seq2.dtype == np.uint8
            assert self.seq2.shape[0] * 4 >= self.qual.shape[0]
        assert self.blk_off[0] == 0 and self.blk_off[-1] == self.n_reads
        for b in range(self.n_blocks):
            s = self.hdr["start"][self.blk_off[b]: self.blk_off[b + 1]]
            assert np.all(s[1:] >= s[:-1]), "read block %d not sorted" % b


def pack_seq(seq_codes: np.ndarray) -> np.ndarray:
    """2-bit pack an array of base codes (values 0..3), base i -> bits 2*(i&3) of byte i>>2."""
    n = seq_codes.shape[0]
    pad = (-n) % 4
    if pad:
        seq_codes = np.concatenate([seq_codes, np.zeros(pad, dtype=seq_codes.dtype)])
    c = seq_codes.astype(np.uint8).reshape(-1, 4)
    return (c[:, 0] | (c[:, 1] << 2) | (c[:, 2] << 4) | (c[:, 3] << 6)).astype(np.uint8)


def encode_bases(seq: str) -> Tuple[np.ndarray, np.ndarray]:
    """ASCII query sequence -> (2-bit codes, escape mask).  Non-ACGT: N -> code 0, other -> 1."""
    b = np.frombuffer(seq.encode("ascii"), dtype=np.uint8)
    code = np.zeros(b.shape[0], dtype=np.uint8)
    esc = np.ones(b.shape[0], dtype=bool)
    for ch, v in BASE2.items():
        m = b == ord(ch)
        code[m] = v
        esc[m] = False
    other = esc & (b != ord("N"))
    code[other] = 1
    return code, esc


def decode_base(code: int, q: int) -> str:
    """Inverse of encode_bases for one base; escaped non-N letters come back as '?'."""
    if q & QUAL_ESCAPE:
        return "N" if code == 0 else "?"
    return BASE_CHARS[code]
