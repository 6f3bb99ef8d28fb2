"""CSI-indexed BCF sites files without cyvcf2: BGZF inflate and CSI region queries on the host, record and genotype
decoding in native code (csrc/bcf.cu), on the GPU with an engine.

* ``BcfFile`` -- one BGZF-compressed BCF 2.2 file and its ``.csi``: the header (samples, the string and contig
  dictionaries, the first record's CHROM for ``get_prefix``) and region queries (``bamio.CsiIndex``; overlap by
  pos0 + rlen as stored, which is the end htslib gives a BCF record).
* ``read_sites`` -- the ``SiteTable`` ``vcfio.read_sites`` returns for the same records written as text, array for
  array.  The records of the union of every interval's chunks are inflated once; record boundaries are walked on the
  host, the fixed fields and the trio members' GT / GQ / AD (or RO / AO) are decoded natively -- on the host, or with
  ``engine=`` on the GPU (``engine.BcfDecoder``), where only the record bytes go up and only the fixed fields and the
  member cells come back.  Interval selection is ``vcfio.select_records``, shared with the text reader.
* ``read_dnms`` -- the DNM dicts ``vcfio.read_dnms`` yields for the same records as text, from a BGZF or uncompressed
  ``.bcf`` read whole.
* ``write_bcf`` -- a sorted ``.bcf`` + ``.csi`` from a ``SiteTable`` with ``vcfio.write_vcf``'s options (tests and tools
  generate their inputs with it).
* ``write_phased_vcf`` -- the phased VCF ``unfazed.write_vcf_output`` writes, from a BCF DNM list: the edit list on the
  host (the core of the text writer, ``vcfio.match_edits``), every record printed as VCF text natively (csrc/bcfout.cu).

The format rules this module assumes (BCF 2.2, VCF specification §6) are listed in DESIGN §5.
"""
from __future__ import annotations

import ctypes as C
import gzip
import os
import re
import struct
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import _lib as L
from .bamio import BgzfReader, CsiIndex, write_bgzf, write_csi
from .packers import build_site_table
from .schema import GT_UNKNOWN, HET, HOM_ALT, HOM_REF, SiteTable
from .vcfio import _records, match_edits, member_columns, phased_header, query_plan, select_records, write_output

MAGIC = b"BCF\x02\x02"
FORMAT_KEYS = ("GT", "GQ", "AD", "RO", "AO")       # the order of UnfzBcfRec.fmt_off
BT_INT8, BT_INT16, BT_INT32, BT_FLOAT, BT_CHAR = 1, 2, 3, 5, 7
_WIDTH = {0: 0, 1: 1, 2: 2, 3: 4, 5: 4, 7: 1}
_INT_LO = {BT_INT8: -128, BT_INT16: -32768, BT_INT32: -(1 << 31)}    # the missing value; end of vector is lo + 1
_FLOAT_MISSING, _FLOAT_EOV = 0x7F800001, 0x7F800002
_BAD_WHY = ((L.BCF_BAD_OVERRUN, "a typed value runs past l_shared / l_indiv"),
            (L.BCF_BAD_SAMPLES, "n_sample differs from the header's sample count"),
            (L.BCF_BAD_TYPE, "unknown type"), (L.BCF_BAD_POS, "POS / rlen out of range"))


def _ptr(a: np.ndarray) -> int:
    return a.ctypes.data


# ------------------------------------------------------------------------------------------------
# native decode on the host (the device decoder, engine.BcfDecoder, has the same two calls)
# ------------------------------------------------------------------------------------------------

def record_offsets(buf: np.ndarray) -> Tuple[np.ndarray, int]:
    """Byte offsets of the records of ``buf`` (walking l_shared + l_indiv from 0) and where the walk stopped; -1 for
    the stop when a record has an l_shared below 24."""
    n = int(buf.shape[0])
    offs = np.empty(n // 32 + 1, dtype=np.int64)
    end = C.c_int64(0)
    got = L.load().unfz_bcf_record_offsets(_ptr(buf), n, offs.shape[0], _ptr(offs), C.byref(end))
    if got < 0:
        return offs[:0], -1 - int(end.value)
    return offs[:got], int(end.value)


class HostDecoder:
    """``records`` and ``samples`` with the host entry points of csrc/bcf.cu."""

    def records(self, buf: np.ndarray, offs: np.ndarray, keys: np.ndarray, n_samples: int) -> np.ndarray:
        """Fixed fields (``_lib.BCF_REC_DTYPE``) of the records at ``offs``."""
        self.buf = buf
        offs = np.ascontiguousarray(offs, dtype=np.int64)
        self.recs = np.empty(offs.shape[0], dtype=L.BCF_REC_DTYPE)
        keys = np.ascontiguousarray(keys, dtype=np.int32)
        if offs.shape[0]:
            L.load().unfz_bcf_parse_host(_ptr(buf), _ptr(offs), int(offs.shape[0]), _ptr(keys), int(n_samples),
                                         _ptr(self.recs))
        return self.recs

    def samples(self, sel: np.ndarray, member_sample: np.ndarray) -> Dict[str, np.ndarray]:
        """Genotype fields of the selected records for the member columns (``member_sample``: column -> sample)."""
        sel = np.ascontiguousarray(sel, dtype=np.int64)
        ms = np.ascontiguousarray(member_sample, dtype=np.int32)
        n, m = sel.shape[0], ms.shape[0]
        out = {"gt": np.empty((n, m), np.uint8), "gq": np.empty((n, m), np.float32), "rd": np.empty((n, m), np.int32),
               "ad": np.empty((n, m), np.int32), "status": np.empty((n, m), np.uint8)}
        if n and m:
            L.load().unfz_bcf_samples_host(_ptr(self.buf), _ptr(self.recs), _ptr(sel), n, _ptr(ms), m,
                                           *(_ptr(out[k]) for k in ("gt", "gq", "rd", "ad", "status")))
        return out

    def format(self, edit_off: np.ndarray, edits: np.ndarray, n_samples: int, names, fkeys: np.ndarray):
        """Every record of ``records()`` printed as the phased VCF body (csrc/bcfout.cu): (the output bytes, the status
        of every record, ``_lib.BCFOUT_*``).  With a haploid phase edit or a malformed record the output is empty."""
        return format_host(self.buf, self.recs, edit_off, edits, n_samples, names, fkeys)[:2]


def format_host(buf, recs, edit_off, edits, n_samples: int, names, fkeys):
    """The host entry points of csrc/bcfout.cu over ``recs``: (output bytes, status of every record, output length of
    every record).  ``names``: (string names, offsets, contig names, offsets) of ``dictionaries``; ``fkeys``: the
    string-dictionary ids of GT, UOPS and UET."""
    lib = L.load()
    n = int(recs.shape[0])
    recs = np.ascontiguousarray(recs, dtype=L.BCF_REC_DTYPE)
    edit_off = np.ascontiguousarray(edit_off, dtype=np.int64)
    edits = np.ascontiguousarray(edits, dtype=L.VCF_EDIT_DTYPE)
    fkeys = np.ascontiguousarray(fkeys, dtype=np.int32)
    sn, so, cn, co = names
    args = (_ptr(buf), _ptr(recs), n, _ptr(sn), _ptr(so), int(so.shape[0]) - 1, _ptr(cn), _ptr(co), int(co.shape[0]) - 1,
            _ptr(fkeys), _ptr(edit_off), _ptr(edits), int(n_samples))
    out_len = np.zeros(max(n, 1), dtype=np.int64)
    status = np.zeros(max(n, 1), dtype=np.uint8)
    total = int(lib.unfz_bcf_format_size_host(*args, _ptr(out_len), _ptr(status)))
    if (status[:n] & (L.BCFOUT_HAPLOID | L.BCFOUT_BAD)).any():
        return np.zeros(0, dtype=np.uint8), status[:n], out_len[:n]
    out_off = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(out_len[:n], out=out_off[1:])
    out = np.empty(total, dtype=np.uint8)
    lib.unfz_bcf_format_write_host(*args, _ptr(out_off), _ptr(out))
    return out, status[:n], out_len[:n]


def _checked_records(dec, buf, offs, keys, n_samples, where) -> np.ndarray:
    recs = dec.records(buf, offs, keys, n_samples)
    bad = np.flatnonzero(recs["flags"] & L.BCF_BAD)
    if bad.shape[0]:
        f = int(recs["flags"][bad[0]])
        why = "; ".join(w for bit, w in _BAD_WHY if f & bit)
        raise ValueError("%s: malformed BCF record (%s)" % (where(int(recs["rec_off"][bad[0]])), why))
    return recs


def _check_cells(cells, recs, sel, where) -> None:
    badc = np.argwhere(cells["status"] & L.BCF_CELL_BAD)
    if badc.shape[0]:
        raise ValueError("%s: malformed genotype field (a reserved value, a wrong type or an overflowing sum)"
                         % where(int(recs["rec_off"][sel[badc[0, 0]]])))


# ------------------------------------------------------------------------------------------------
# header
# ------------------------------------------------------------------------------------------------

_HREC = re.compile(r"^##(FILTER|INFO|FORMAT|contig)=<(.*)>\s*$")


def _hrec_fields(body: str) -> Dict[str, str]:
    """key=value pairs of a structured header line; quoted values may hold commas."""
    out, i, n = {}, 0, len(body)
    while i < n:
        j = body.find("=", i)
        if j < 0:
            break
        key = body[i:j].strip()
        k = j + 1
        if k < n and body[k] == '"':
            k += 1
            while k < n and body[k] != '"':
                k += 2 if body[k] == "\\" else 1
            val, k = body[j + 2:k], k + 1
        else:
            e = body.find(",", k)
            e = n if e < 0 else e
            val, k = body[k:e], e
        out.setdefault(key, val)
        i = k + 1                                    # past the comma
    return out


def parse_header(text: str, path: str):
    """(samples, string dictionary ID -> index, contig names by index) of a BCF header text.  The string dictionary
    holds FILTER, INFO and FORMAT IDs in one namespace: PASS is 0, ``IDX=`` sets an index, and otherwise IDs are numbered
    by first appearance after the highest index so far; the contig dictionary likewise holds the ``##contig`` lines."""
    strs: Dict[str, int] = {"PASS": 0}
    n_str = 1
    contigs: Dict[str, int] = {}
    n_ctg = 0
    samples: Optional[List[str]] = None
    for line in text.split("\n"):
        if line.startswith("#CHROM"):
            samples = line.rstrip("\r").split("\t")[9:]
            break
        m = _HREC.match(line)
        if not m:
            continue
        f = _hrec_fields(m.group(2))
        ident = f.get("ID")
        if ident is None:
            continue
        idx = f.get("IDX")
        try:
            idx = int(idx) if idx is not None else None
        except ValueError:
            raise ValueError("%s: header line with IDX=%r" % (path, idx))
        if m.group(1) == "contig":
            if ident not in contigs:
                contigs[ident] = n_ctg if idx is None else idx
                n_ctg = max(n_ctg, contigs[ident] + 1)
        elif ident not in strs:
            strs[ident] = n_str if idx is None else idx
            n_str = max(n_str, strs[ident] + 1)
    if samples is None:
        raise ValueError("%s: no #CHROM header line" % path)
    names = [""] * n_ctg
    for c, i in contigs.items():
        names[i] = c
    return samples, strs, names


def _read_head(data: bytes, path: str):
    """(header text, offset of the first record) of the start of an inflated BCF; None when ``data`` is too short."""
    if len(data) >= 5 and data[:5] != MAGIC:
        raise ValueError("%s: not a BCF 2.2 file (magic %r)" % (path, data[:5]))
    if len(data) < 9:
        return None
    l_text = struct.unpack_from("<I", data, 5)[0]
    if len(data) < 9 + l_text:
        return None
    return data[9:9 + l_text].split(b"\0", 1)[0].decode("utf-8", "replace"), 9 + l_text


def index_path(path: str) -> Optional[str]:
    """``<file>.csi`` if it exists."""
    p = path + ".csi"
    return p if os.path.exists(p) else None


class BcfFile:
    """One BGZF-compressed, CSI-indexed BCF 2.2 file: header and region queries."""

    def __init__(self, path: str, index: Optional[str] = None):
        self.path = path
        self.bgzf = BgzfReader(path)
        ip = index or index_path(path)
        if ip is None:
            raise ValueError("%s: no .csi index" % path)
        self.csi = CsiIndex(ip)
        want = 1 << 16
        while True:
            head, eof = self.bgzf.stream_from(0, want)
            hb = head.tobytes()
            got = _read_head(hb, path)
            if got is not None and (len(hb) >= got[1] + 12 or eof):
                break
            if eof:
                raise ValueError("%s: truncated BCF header" % path)
            want = 4 * len(hb)
        text, first = got
        self.samples, self.strings, self.contigs = parse_header(text, path)
        self.tids = {c: i for i, c in enumerate(self.contigs) if c}
        self.keys = np.array([self.strings.get(k, -1) for k in FORMAT_KEYS], dtype=np.int32)
        chrom = None
        if len(hb) >= first + 12:
            cid = struct.unpack_from("<i", hb, first + 8)[0]
            chrom = self.contigs[cid] if 0 <= cid < len(self.contigs) else None
        self.prefix = "" if chrom is None or "chr" not in chrom.lower() else chrom[:3]

    def fetch_union(self, queries: Sequence[Tuple[int, int, int]]):
        """Inflated records of the union of the chunk lists of many (tid, beg, end) queries, their offsets, and a
        function that names a byte of the buffer (the file and the virtual offset of its chunk plus the bytes after it)
        for error messages."""
        ch = sorted(c for tid, beg, end in queries for c in self.csi.chunks(tid, beg, end))
        merged: List[List[int]] = []
        for b, e in ch:
            if merged and b <= merged[-1][1]:
                merged[-1][1] = max(merged[-1][1], e)
            else:
                merged.append([b, e])
        parts = self.bgzf.read_ranges([(b, e) for b, e in merged])
        offs, base = [], 0
        for (vb, _), p in zip(merged, parts):
            o, stop = record_offsets(p)
            if stop < 0:
                raise ValueError("%s, record at virtual offset %d + %d bytes: malformed BCF record (l_shared below 24)"
                                 % (self.path, vb, -1 - stop))
            if stop != p.shape[0]:
                raise ValueError("%s: the CSI chunk at virtual offset %d does not end on a record boundary"
                                 % (self.path, vb))
            offs.append(o + base)
            base += p.shape[0]
        starts = np.cumsum([0] + [p.shape[0] for p in parts])
        buf = np.concatenate(parts) if parts else np.zeros(0, dtype=np.uint8)
        offs = np.concatenate(offs) if offs else np.zeros(0, dtype=np.int64)

        def where(off: int):
            k = int(np.searchsorted(starts, off, side="right")) - 1
            return "%s, record at virtual offset %d + %d bytes" % (self.path, merged[k][0], off - int(starts[k]))
        return buf, offs, where

    def query(self, contig: str, beg: int, end: int) -> np.ndarray:
        """Fixed fields of the records overlapping [beg, end) of contig, in file order (host decode)."""
        tid = self.tids.get(contig)
        if tid is None:
            return np.zeros(0, dtype=L.BCF_REC_DTYPE)
        buf, offs, where = self.fetch_union([(tid, beg, end)])
        recs = _checked_records(HostDecoder(), buf, offs, self.keys, len(self.samples), where)
        keep = (recs["contig"] == tid) & (recs["pos0"] < end) & (recs["rend"] > beg)
        return recs[keep]


# ------------------------------------------------------------------------------------------------
# site reader
# ------------------------------------------------------------------------------------------------

def _typed(b: np.ndarray, p: int) -> Tuple[int, int, int]:
    """(type, count, offset of the first value) of the typed value at byte p."""
    t = int(b[p])
    ty, n = t & 15, t >> 4
    p += 1
    if n == 15:
        ct = int(b[p]) & 15
        w = _WIDTH[ct]
        n = int(b[p + 1: p + 1 + w].view({1: "<i1", 2: "<i2", 4: "<i4"}[w])[0])
        p += 1 + w
    return ty, n, p


def _alleles(buf: np.ndarray, rec) -> List[str]:
    """Every allele string of a record (REF first), NUL padding dropped."""
    o = int(rec["rec_off"])
    _t, n, p = _typed(buf, o + 32)                   # ID
    p += n
    out = []
    for _ in range(int(rec["n_allele"])):
        _t, n, p = _typed(buf, p)
        out.append(buf[p:p + n].tobytes().rstrip(b"\0").decode())
        p += n
    return out


def read_sites(path, trios: Sequence[Tuple[str, str, str]], regions: Dict[str, List[Tuple[int, int]]],
               engine=None) -> SiteTable:
    """``vcfio.read_sites`` of the same records as text, from the BCF directly.  ``path``: a file name or a
    ``BcfFile``.  With ``engine`` the records are decoded on that engine's GPU (``Engine.bcf_decoder``)."""
    bf = path if isinstance(path, BcfFile) else BcfFile(path)
    slot_of, n_members, cols = member_columns(bf.samples, trios)
    member_sample = np.zeros(n_members, dtype=np.int32)
    member_sample[slot_of[slot_of >= 0]] = np.flatnonzero(slot_of >= 0)
    plan, queries = query_plan(regions, bf.tids)
    buf, offs, where = bf.fetch_union(queries)
    dec = engine.bcf_decoder() if engine is not None else HostDecoder()
    recs = _checked_records(dec, buf, offs, bf.keys, len(bf.samples), where)
    pos0 = recs["pos0"].astype(np.int64)
    sel, cid, contigs = select_records(plan, recs["contig"].astype(np.int64), pos0, recs["rend"].astype(np.int64))
    r = recs[sel]
    simple = (r["flags"] & L.BCF_SIMPLE) != 0
    alt_b = np.zeros(sel.shape[0], dtype=np.uint8)
    has_alt = (r["n_allele"] > 1) & (r["alt_len"] > 0)
    alt_b[has_alt] = buf[(r["rec_off"] + r["alt_off"])[has_alt]]
    refalt = {}
    for i in np.flatnonzero(~simple).tolist():
        al = _alleles(buf, r[i])
        refalt[i] = (al[0] if al else "", al[1:])
    cells = dec.samples(sel, member_sample)
    _check_cells(cells, recs, sel, where)
    return build_site_table(trios, cols, contigs, cid, pos0[sel], simple, r["ref0"].astype(np.uint8), alt_b,
                            cells["gt"], cells["gq"], cells["rd"], cells["ad"], refalt)


# ------------------------------------------------------------------------------------------------
# DNM reader
# ------------------------------------------------------------------------------------------------

def _info_string(buf: np.ndarray, rec, key: int) -> Optional[str]:
    """The INFO value of dictionary key ``key`` as a string (None: absent)."""
    o = int(rec["rec_off"])
    _t, n, p = _typed(buf, o + 32)                   # ID
    p += n
    for _ in range(int(rec["n_allele"])):
        _t, n, p = _typed(buf, p)
        p += n
    t, n, p = _typed(buf, p)                         # FILTER
    p += n * _WIDTH[t]
    n_info = int(buf[o + 24: o + 28].view("<u4")[0]) & 0xFFFF
    for _ in range(n_info):
        t, n, p = _typed(buf, p)
        k = int(buf[p: p + _WIDTH[t]].view({1: "<i1", 2: "<i2", 4: "<i4"}[_WIDTH[t]])[0])
        p += _WIDTH[t]
        t, n, p = _typed(buf, p)
        if k == key:
            return buf[p:p + n].tobytes().split(b"\0", 1)[0].decode() if t == BT_CHAR else None
        p += n * _WIDTH.get(t, 0)
    return None


def _read_whole(path: str):
    """A BGZF-compressed or uncompressed BCF read whole: (header text, samples, string dictionary, contig names, the
    record bytes (writable), their offsets, and a function that names a byte of them for error messages)."""
    with open(path, "rb") as f:
        bgzf = f.read(2) == b"\x1f\x8b"
    if bgzf:
        BgzfReader(path)                             # the EOF block check
    with (gzip.open if bgzf else open)(path, "rb") as f:
        data = bytearray().join(iter(lambda: f.read(1 << 24), b""))
    got = _read_head(data, path)
    if got is None:
        raise ValueError("%s: truncated BCF header" % path)
    text, first = got
    samples, strs, contigs = parse_header(text, path)
    buf = np.frombuffer(data, dtype=np.uint8)[first:]
    where = lambda off: "%s, record at byte %d" % (path, first + off)
    offs, stop = record_offsets(buf)
    if stop < 0 or stop != buf.shape[0]:
        raise ValueError("%s: malformed or truncated BCF record" % where(stop if stop >= 0 else -1 - stop))
    return text, samples, strs, contigs, buf, offs, where


def is_bcf(path: str) -> bool:
    """``path`` holds BCF 2.2, uncompressed or BGZF-compressed (by its magic)."""
    with open(path, "rb") as f:
        head = f.read(5)
    if head[:2] == b"\x1f\x8b":
        try:
            with gzip.open(path, "rb") as g:
                head = g.read(5)
        except (OSError, EOFError):
            return False
    return head == MAGIC


def read_dnms(path: str):
    """The DNMs of a BGZF-compressed or uncompressed BCF, read whole without an index: for every record and every
    sample whose genotype is HET or HOM_ALT, in header order, {chrom, start, end, kid, vartype, bam: ""} with start
    pos0, end pos0 + rlen and vartype INFO SVTYPE or "POINT" -- what ``vcfio.read_dnms`` yields for the same records as
    text."""
    from .utils import SNV_TYPES
    _text, samples, strs, contigs, buf, offs, where = _read_whole(path)
    dec = HostDecoder()
    keys = np.array([strs.get(k, -1) for k in FORMAT_KEYS], dtype=np.int32)
    recs = _checked_records(dec, buf, offs, keys, len(samples), where)
    sel = np.arange(recs.shape[0], dtype=np.int64)
    cells = dec.samples(sel, np.arange(len(samples), dtype=np.int32))
    _check_cells(cells, recs, sel, where)
    gt = cells["gt"]
    sv_key = strs.get("SVTYPE", -1)
    for i in range(recs.shape[0]):
        carriers = np.flatnonzero((gt[i] == HET) | (gt[i] == HOM_ALT)).tolist()
        if not carriers:
            continue
        vartype = (_info_string(buf, recs[i], sv_key) if sv_key >= 0 else None) or SNV_TYPES[0]
        cid = int(recs["contig"][i])
        if not 0 <= cid < len(contigs):
            raise ValueError("%s: CHROM %d is not in the contig dictionary" % (where(int(recs["rec_off"][i])), cid))
        for s in carriers:
            yield {"chrom": contigs[cid], "start": int(recs["pos0"][i]), "end": int(recs["rend"][i]),
                   "kid": samples[s], "vartype": vartype, "bam": ""}


# ------------------------------------------------------------------------------------------------
# phased VCF writer
# ------------------------------------------------------------------------------------------------

_IDX = re.compile(r",IDX=[0-9]+(?=[,>])")


def vcf_header(text: str) -> str:
    """The header text of a BCF as VCF: ``IDX=`` dropped from the dictionary lines (htslib writes it to BCF only)."""
    return "\n".join(_IDX.sub("", x) if _HREC.match(x) else x for x in text.split("\n"))


def dictionaries(strs: Dict[str, int], contigs: Sequence[str]):
    """The string dictionary and the contig dictionary as names for csrc/bcfout.cu: (string names, int64 offsets,
    contig names, int64 offsets); an unused index has an empty name."""
    by_id = [""] * (max(strs.values()) + 1 if strs else 0)
    for k, i in strs.items():
        by_id[i] = k
    out = []
    for names in (by_id, list(contigs)):
        b = [x.encode() for x in names]
        off = np.zeros(len(b) + 1, dtype=np.int64)
        np.cumsum([len(x) for x in b], out=off[1:])
        out += [np.frombuffer(b"".join(b) + b"\0", dtype=np.uint8), off]
    return tuple(out)


def phase_edits(buf: np.ndarray, recs: np.ndarray, samples: Sequence[str], strs: Dict[str, int], contigs: Sequence[str],
                read_records, include_ambiguous, verbose, evidence_min_ratio, dec=None):
    """``vcfio.match_edits`` of the records of a BCF DNM list: CHROM from the contig dictionary, SVTYPE from INFO, the
    kids' genotypes from the decoder's ``samples``."""
    from .utils import SNV_TYPES
    dec = dec or HostDecoder()
    sv_key = strs.get("SVTYPE", -1)

    def chrom_of(i):
        cid = int(recs["contig"][i])
        return contigs[cid] if 0 <= cid < len(contigs) else None

    def svtype_of(i):
        return (_info_string(buf, recs[i], sv_key) if sv_key >= 0 else None) or SNV_TYPES[0]
    return match_edits(recs["pos0"], recs["rend"], chrom_of, svtype_of,
                       lambda sel, kids: dec.samples(sel, np.asarray(kids, dtype=np.int32))["gt"], samples, read_records,
                       include_ambiguous, verbose, evidence_min_ratio)


def write_phased_vcf(in_path: str, read_records, include_ambiguous, verbose, outfile: str, evidence_min_ratio,
                     engine=None) -> None:
    """The phased VCF of ``unfazed.write_vcf_output`` from a BCF 2.2 DNM list (BGZF or uncompressed) without cyvcf2:
    every record printed as htslib's vcf_format prints it, with GT 1|0 (paternal) / 0|1 (maternal) and UOPS / UET for
    the phased carriers, UOPS = UET = -1 in every other cell.  The edit list is built on the host (``phase_edits``); the
    records are printed in native code (csrc/bcfout.cu), on ``engine``'s GPU when given.  The header is the BCF's with
    ``IDX=`` dropped, plus the lines ``vcfio.phased_header`` adds.  ``outfile``: ``/dev/stdout`` or a plain file, BGZF
    when it ends in ``.gz``."""
    from . import __version__
    text, samples, strs, contigs, buf, offs, where = _read_whole(in_path)
    dec = engine.bcf_decoder() if engine is not None else HostDecoder()
    keys = np.array([strs.get(k, -1) for k in FORMAT_KEYS], dtype=np.int32)
    recs = _checked_records(dec, buf, offs, keys, len(samples), where)
    edit_off, edits = phase_edits(buf, recs, samples, strs, contigs, read_records, include_ambiguous, verbose,
                                  evidence_min_ratio, dec)
    names = dictionaries(strs, contigs)
    fkeys = np.array([strs.get(k, -1) for k in ("GT", "UOPS", "UET")], dtype=np.int32)
    out, status = dec.format(edit_off, edits, len(samples), names, fkeys)
    bad = np.flatnonzero(status & (L.BCFOUT_HAPLOID | L.BCFOUT_BAD))
    if bad.shape[0]:
        i = int(bad[0])
        off = int(recs["rec_off"][i])
        if status[i] & L.BCFOUT_BAD:
            raise ValueError("%s: malformed BCF record (an id outside the header's dictionaries, or a value of a type it "
                             "cannot have)" % where(off))
        # the record printed without edits names the GT
        line, _, _ = format_host(buf, recs[i:i + 1], np.zeros(2, dtype=np.int64), edits[:0], len(samples), names, fkeys)
        cols = line.tobytes().decode("utf-8", "replace").rstrip("\n").split("\t")
        gi = cols[8].split(":").index("GT")
        e = edits[int(edit_off[i]): int(edit_off[i + 1])]
        for s in e["sample"][e["phase"] != 0].tolist():
            gt = cols[9 + s].split(":")[gi]
            if "/" not in gt and "|" not in gt:
                raise ValueError("%s: the haploid GT %r of sample %s cannot be phased" % (where(off), gt, samples[s]))
    write_output(outfile, phased_header(vcf_header(text).encode(), __version__), out)


# ------------------------------------------------------------------------------------------------
# writer
# ------------------------------------------------------------------------------------------------

_MISS = np.iinfo(np.int64).min                       # missing / end-of-vector markers of the writer's int64 arrays
_EOV = _MISS + 1
_GT_CODES = {HOM_REF: (2, 2), HET: (2, 4), HOM_ALT: (4, 4), GT_UNKNOWN: (0, 0)}     # (allele + 1) << 1, unphased


def _typed_hdr(ty: int, n: int) -> bytes:
    if n < 15:
        return bytes([(n << 4) | ty])
    return bytes([0xF0 | ty]) + _typed_int(n)


def _typed_int(v: int) -> bytes:
    """One integer as a typed value of the narrowest width."""
    ty, vals = _int_vec(np.array([v], dtype=np.int64))
    return bytes([0x10 | ty]) + vals


def _int_vec(v: np.ndarray) -> Tuple[int, bytes]:
    """(type, bytes) of an int64 array with _MISS / _EOV markers, in the narrowest integer type that holds its values
    above the reserved range (htslib's bcf_enc_vint)."""
    real = v[(v != _MISS) & (v != _EOV)]
    lo, hi = (int(real.min()), int(real.max())) if real.shape[0] else (0, 0)
    if -120 <= lo and hi <= 127:
        ty, dt = BT_INT8, "<i1"
    elif -32760 <= lo and hi <= 32767:
        ty, dt = BT_INT16, "<i2"
    else:
        ty, dt = BT_INT32, "<i4"
    base = _INT_LO[ty]
    out = np.where(v == _MISS, base, np.where(v == _EOV, base + 1, v))
    return ty, out.astype(dt).tobytes()


def _string(s: str) -> bytes:
    b = s.encode()
    return _typed_hdr(BT_CHAR, len(b)) + b


def write_bcf(table: SiteTable, path: str, end: Optional[Dict[int, int]] = None,
              format_order: Optional[Sequence[Sequence[str]]] = None, level: int = 6, min_shift: int = 14,
              depth: Optional[int] = None) -> None:
    """Sorted ``path`` (.bcf, BGZF) + ``path.csi`` of ``table``: the records ``vcfio.write_vcf`` writes, in BCF 2.2.
    Every sample of every trio; GT / AD / GQ missing for a trio without a row in the record.  GQ is Float when a value is
    not integral, else an integer; integers take the narrowest width that holds a field's values, as htslib chooses
    them.  The header carries ``IDX=`` on its dictionary lines, as htslib writes it.  ``end``: record index -> INFO END
    (1-based inclusive; rlen = END - pos0); ``format_order``: record index -> the order of GT / AD / GQ.  CSI of
    ``min_shift`` / ``depth`` (None: the smallest depth that spans the records)."""
    t = table
    view_rows, g_lo, g_contig = _records(t)
    n_rec = g_lo.shape[0] - 1
    samples: List[str] = []
    for trio in t.trios:
        for s in trio:
            if s not in samples:
                samples.append(s)
    sidx = {s: i for i, s in enumerate(samples)}
    ns = len(samples)
    blk = np.repeat(np.arange(t.n_blocks), np.diff(t.blk_off))
    is_float = bool(np.any((t.gq != np.round(t.gq)) & (t.gq != -1)))
    key = {"PASS": 0, "END": 1, "GT": 2, "AD": 3, "GQ": 4}
    head = ["##fileformat=VCFv4.2", '##FILTER=<ID=PASS,Description="All filters passed",IDX=0>']
    head += ["##contig=<ID=%s,IDX=%d>" % (c, i) for i, c in enumerate(t.contigs)]
    head += ['##INFO=<ID=END,Number=1,Type=Integer,Description="End position",IDX=1>',
             '##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype",IDX=2>',
             '##FORMAT=<ID=AD,Number=R,Type=Integer,Description="Allelic depths",IDX=3>',
             '##FORMAT=<ID=GQ,Number=1,Type=%s,Description="Genotype quality",IDX=4>' % ("Float" if is_float else "Integer"),
             "\t".join(["#CHROM", "POS", "ID", "REF", "ALT", "QUAL", "FILTER", "INFO", "FORMAT"] + samples)]
    text = ("\n".join(head) + "\n").encode() + b"\0"
    head_b = MAGIC + struct.pack("<I", len(text)) + text
    recs: List[bytes] = []
    pos0 = np.zeros(n_rec, dtype=np.int64)
    rend = np.zeros(n_rec, dtype=np.int64)
    for g in range(n_rec):
        rows = view_rows[g_lo[g]: g_lo[g + 1]]
        lead = int(rows[0])
        ref, alts = t.ref_alts(lead)
        p0 = int(t.pos[lead])
        order = tuple(format_order[g]) if format_order is not None else ("GT", "AD", "GQ")
        gt = np.zeros((ns, 2), dtype=np.int64)
        ad = np.full((ns, 2), _MISS, dtype=np.int64)
        ad[:, 1] = _EOV
        gq = np.full(ns, -1.0, dtype=np.float32)
        for row in rows.tolist():
            tr = t.trios[int(t.blk_trio[blk[row]])]
            for m in range(3):
                s = sidx[tr[m]]
                gt[s] = _GT_CODES[int(t.gt[m, row])]
                rd_, ad_ = int(t.rd[m, row]), int(t.ad[m, row])
                if not (rd_ == -1 and ad_ == -1):
                    ad[s] = (_MISS if rd_ == -1 else rd_, _MISS if ad_ == -1 else ad_)
                gq[s] = t.gq[m, row]
        fields = {}
        ty, vals = _int_vec(gt.reshape(-1))
        fields["GT"] = _typed_hdr(ty, 2) + vals
        ty, vals = _int_vec(ad.reshape(-1))
        fields["AD"] = _typed_hdr(ty, 2) + vals
        if is_float:
            bits = gq.view(np.uint32).copy()
            bits[gq == -1] = _FLOAT_MISSING
            fields["GQ"] = _typed_hdr(BT_FLOAT, 1) + bits.astype("<u4").tobytes()
        else:
            ty, vals = _int_vec(np.where(gq == -1, _MISS, gq.astype(np.int64)))
            fields["GQ"] = _typed_hdr(ty, 1) + vals
        indiv = b"".join(_typed_int(key[k]) + fields[k] for k in order)
        e = (end or {}).get(g)
        r_end = e if (e is not None and e > p0) else p0 + len(ref)
        info = (_typed_int(key["END"]) + _typed_int(e)) if e is not None else b""
        alleles = [ref] + list(alts)
        shared = (struct.pack("<iiiIII", int(g_contig[g]), p0, r_end - p0, _FLOAT_MISSING,
                              (len(alleles) << 16) | (1 if e is not None else 0), (len(order) << 24) | ns)
                  + _string(".") + b"".join(_string(a) for a in alleles) + _typed_hdr(BT_INT8, 1) + b"\0" + info)
        recs.append(struct.pack("<II", len(shared), len(indiv)) + shared + indiv)
        pos0[g] = p0
        rend[g] = r_end
    body = b"".join(recs)
    starts = np.cumsum([0] + [len(x) for x in recs]).astype(np.int64)
    voff = write_bgzf(path, head_b, body, level)
    write_csi(path + ".csi", len(t.contigs), g_contig.astype(np.int64), pos0, rend, voff(starts[:-1]),
              voff(starts[1:]), min_shift=min_shift, depth=depth, level=level)
