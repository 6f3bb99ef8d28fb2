"""Tabix-indexed sites VCFs without cyvcf2: BGZF inflate and TBI region queries on the host, field decoding in native
code (csrc/vcf.cu), on the GPU with an engine.

* ``VcfFile`` -- one bgzipped VCF and its ``.tbi`` or ``.csi``: the header (sample names, the declared Type of the GQ / AD / RO /
  AO FORMAT fields, the first record's CHROM for ``get_prefix``) and region queries (``TbiIndex``: the BAI bins, chunks
  and linear index behind a tabix header, read by ``bamio``'s code; overlap by tabix's end, INFO END or POS + len(REF)).
* ``read_sites`` -- the ``SiteTable`` ``packers.pack_sites`` builds from a cyvcf2 handle over the same regions, array
  for array.  The text of the union of every interval's chunks is inflated once; line boundaries, fixed fields and the
  genotype fields of the trio members are decoded natively -- on the host, or with ``engine=`` on the GPU
  (``engine.VcfDecoder``), where only the text goes up and only the fixed fields and member columns come back.
* ``read_dnms`` -- the DNM dicts ``unfazed.read_vars_vcf`` yields, from a plain or gzipped VCF read whole.
* ``write_vcf`` -- a sorted ``.vcf.gz`` + ``.tbi`` from a ``SiteTable`` (tests and tools generate their inputs with it).
* ``write_phased_vcf`` -- the phased VCF ``unfazed.write_vcf_output`` writes, from a plain or gzipped DNM VCF: the
  edit list of the phased cells on the host, the sample columns rewritten natively (csrc/vcfout.cu).

Field decoding follows cyvcf2 0.31.0's defaults (gts012=False, strict_gt=False); DESIGN §5 lists the assumptions.  A
``.csi`` index (``bamio.CsiIndex``, with the tabix header in its aux bytes) serves where no ``.tbi`` exists.  BCF is read
by ``bcfio``, which shares the interval selection (``select_records``); unindexed files go to cyvcf2.
"""
from __future__ import annotations

import gzip
import os
import re
import struct
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import _lib as L
from .bamio import BaiIndex, BgzfReader, CsiIndex, index_refs, parse_bins, write_bgzf, write_csi
from .packers import _merge, build_site_table
from .schema import GT_UNKNOWN, HET, HOM_ALT, HOM_REF, SiteTable

FAST_DIGITS = 15                 # significant digits of a float GQ decoded in native code (the exact fast path)


def _ptr(a: np.ndarray) -> int:
    return a.ctypes.data


# ------------------------------------------------------------------------------------------------
# native decode on the host (the device decoder, engine.VcfDecoder, has the same calls)
# ------------------------------------------------------------------------------------------------

class HostDecoder:
    """``lines`` and ``samples`` with the host entry points of csrc/vcf.cu, ``rewrite`` with those of csrc/vcfout.cu."""

    def lines(self, buf: np.ndarray) -> np.ndarray:
        """Fixed fields (``_lib.VCF_REC_DTYPE``) of every '\\n'-terminated line of ``buf``."""
        self.buf = buf
        lib = L.load()
        cap = int(np.count_nonzero(buf == 10))
        ends = np.empty(max(cap, 1), dtype=np.int64)
        n = lib.unfz_vcf_line_ends_host(_ptr(buf), int(buf.shape[0]), cap, _ptr(ends))
        self.recs = np.empty(n, dtype=L.VCF_REC_DTYPE)
        if n:
            lib.unfz_vcf_parse_host(_ptr(buf), _ptr(ends), n, _ptr(self.recs))
        return self.recs

    def samples(self, sel: np.ndarray, slot_of: np.ndarray, n_members: int, gq_float: bool,
                max_digits: int = FAST_DIGITS) -> Dict[str, np.ndarray]:
        """Genotype fields of the selected lines for the member columns (``slot_of``: sample -> column or -1)."""
        sel = np.ascontiguousarray(sel, dtype=np.int64)
        slot_of = np.ascontiguousarray(slot_of, dtype=np.int32)
        out = _empty_cells(sel.shape[0], n_members)
        L.load().unfz_vcf_samples_host(_ptr(self.buf), _ptr(self.recs), _ptr(sel), int(sel.shape[0]), _ptr(slot_of),
                                       int(slot_of.shape[0]), int(n_members), int(bool(gq_float)), int(max_digits),
                                       *(_ptr(out[k]) for k in ("gt", "gq", "rd", "ad", "status", "line_bad")))
        return out

    def rewrite(self, edit_off: np.ndarray, edits: np.ndarray, n_samples: int):
        """Every line of ``lines()`` rewritten with the edit list (``_lib.VCF_EDIT_DTYPE``, CSR by line): (the output
        bytes, the status of every line, ``_lib.VCFOUT_*``).  With a bad line the output is empty."""
        lib = L.load()
        n = int(self.recs.shape[0])
        edit_off = np.ascontiguousarray(edit_off, dtype=np.int64)
        edits = np.ascontiguousarray(edits, dtype=L.VCF_EDIT_DTYPE)
        out_len = np.empty(max(n, 1), dtype=np.int64)
        line_bad = np.zeros(max(n, 1), dtype=np.uint8)
        args = (_ptr(self.buf), _ptr(self.recs), n, _ptr(edit_off), _ptr(edits), int(n_samples))
        total = int(lib.unfz_vcf_rewrite_size_host(*args, _ptr(out_len), _ptr(line_bad)))
        if line_bad[:n].any():
            return np.zeros(0, dtype=np.uint8), line_bad[:n]
        out_off = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(out_len[:n], out=out_off[1:])
        out = np.empty(total, dtype=np.uint8)
        lib.unfz_vcf_rewrite_write_host(*args, _ptr(out_off), _ptr(out))
        return out, line_bad[:n]


def _empty_cells(n: int, m: int) -> Dict[str, np.ndarray]:
    return {"gt": np.empty((n, m), np.uint8), "gq": np.empty((n, m), np.float32), "rd": np.empty((n, m), np.int32),
            "ad": np.empty((n, m), np.int32), "status": np.empty((n, m), np.uint8), "line_bad": np.empty(n, np.uint8)}


def _field_end(text: np.ndarray, a: int) -> int:
    e = a
    while e < text.shape[0] and text[e] not in (9, 10, 13, 58):      # tab, newline, CR, ':'
        e += 1
    return e


def finish_cells(cells: Dict[str, np.ndarray], buf: np.ndarray, recs: np.ndarray, sel: np.ndarray, where) -> None:
    """Raises ``ValueError`` for malformed fields; decodes on the host the float GQs the native code left to it (their
    cell holds the int32 offset of the text from the line start) with Python's correctly rounded ``float``, then cast
    to float32 -- what htslib's strtod-to-float gives."""
    bad = np.flatnonzero(cells["line_bad"])
    if bad.shape[0]:
        raise ValueError("%s: more sample columns than header samples" % where(int(recs["line_off"][sel[bad[0]]])))
    st = cells["status"]
    badc = np.argwhere(st & L.VCF_CELL_BAD)
    if badc.shape[0]:
        raise ValueError("%s: malformed or overflowing genotype field" % where(int(recs["line_off"][sel[badc[0, 0]]])))
    host = np.argwhere(st & L.VCF_CELL_HOST)
    if host.shape[0]:
        gq = cells["gq"]
        offs = gq.view(np.int32)
        for i, m in host.tolist():
            a = int(recs["line_off"][sel[i]]) + int(offs[i, m])
            txt = buf[a:_field_end(buf, a)].tobytes().decode("ascii", "replace")
            try:
                gq[i, m] = np.float32(float(txt))
            except ValueError:
                raise ValueError("%s: GQ %r is not a number" % (where(a), txt))


# ------------------------------------------------------------------------------------------------
# TBI
# ------------------------------------------------------------------------------------------------

class TbiIndex(BaiIndex):
    """A tabix index: the reference names of its header, then bins, chunks and linear index laid out as BAI's (the
    region queries are ``BaiIndex.chunks``)."""

    def __init__(self, path: str):
        raw, _ = BgzfReader(path).stream_from(0, 1 << 62)
        d = raw.tobytes()
        if d[:4] != b"TBI\x01":
            raise ValueError("%s: not a TBI index" % path)
        n_ref, _fmt, _cs, _cb, _ce, _meta, _skip, l_nm = struct.unpack_from("<8i", d, 4)
        self.names = [x.decode() for x in d[36:36 + l_nm].split(b"\0")[:n_ref]]
        self.bins, self.linear, _ = parse_bins(d, 36 + l_nm, n_ref)


def index_path(path: str) -> Optional[str]:
    """``<file>.tbi`` if it exists, else ``<file>.csi`` if it exists."""
    for p in (path + ".tbi", path + ".csi"):
        if os.path.exists(p):
            return p
    return None


def open_tabix_index(path: str):
    """The TBI or CSI index of a bgzipped VCF; both carry the tabix header with the reference names."""
    if path.endswith(".csi"):
        idx = CsiIndex(path)
        if idx.names is None:
            raise ValueError("%s: a CSI index without a tabix header cannot index a VCF" % path)
        return idx
    return TbiIndex(path)


# ------------------------------------------------------------------------------------------------
# VCF file
# ------------------------------------------------------------------------------------------------

_FORMAT_RE = re.compile(rb"^##FORMAT=<ID=([^,>]+),.*?Type=([A-Za-z]+)")


def _prefix_of(chrom: Optional[str]) -> str:
    """``utils.get_prefix`` on a first record of this CHROM (None: no record)."""
    if chrom is None or "chr" not in chrom.lower():
        return ""
    return chrom[:3]


def _parse_header(text: bytes, path: str):
    """(samples, FORMAT types, first CHROM or None, offset of the first data line) of a VCF whose text starts with
    ``text``; None when ``text`` ends before the #CHROM line and the line after it are complete."""
    i = 0 if text.startswith(b"#CHROM") else text.find(b"\n#CHROM") + 1
    if i <= 0 and not text.startswith(b"#CHROM"):
        return None
    j = text.find(b"\n", i)
    if j < 0:
        return None
    k = text.find(b"\n", j + 1)
    cols = text[i:j].rstrip(b"\r").decode().split("\t")
    if len(cols) < 8:
        raise ValueError("%s: malformed #CHROM header line" % path)
    types = {}
    for line in text[:i].split(b"\n"):
        m = _FORMAT_RE.match(line)
        if m:
            types[m.group(1).decode()] = m.group(2).decode()
    first = text[j + 1:k if k >= 0 else len(text)]
    chrom = first.split(b"\t", 1)[0].decode() if first.strip() else None
    return cols[9:], types, chrom, j + 1, k >= 0


class VcfFile:
    """One bgzipped VCF indexed by a TBI or a CSI: header and region queries."""

    def __init__(self, path: str, index: Optional[str] = None):
        self.path = path
        self.bgzf = BgzfReader(path)
        ip = index or index_path(path)
        if ip is None:
            raise ValueError("%s: no .tbi or .csi index" % path)
        self.tbi = open_tabix_index(ip)
        self.tids = {n: i for i, n in enumerate(self.tbi.names)}
        want = 1 << 16
        while True:
            head, eof = self.bgzf.stream_from(0, want)
            hb = head.tobytes()
            got = _parse_header(hb, path)
            if got is not None and (got[4] or eof):
                break
            if eof:
                raise ValueError("%s: no #CHROM header line" % path)
            want = 4 * len(hb)
        self.samples, self.format_types, chrom, _, _ = got
        self.prefix = _prefix_of(chrom)

    def gq_float(self) -> bool:
        """GQ is decoded as a float unless the header declares it Integer."""
        return self.format_types.get("GQ", "Float") != "Integer"

    def fetch_union(self, queries: Sequence[Tuple[int, int, int]]):
        """Inflated text of the union of the chunk lists of many (tid, beg, end) queries, and a function that names a
        byte of it (the file and the virtual offset of its chunk plus the bytes after it) for error messages."""
        ch = sorted(c for tid, beg, end in queries for c in self.tbi.chunks(tid, beg, end))
        merged: List[List[int]] = []
        for b, e in ch:
            if merged and b <= merged[-1][1]:
                merged[-1][1] = max(merged[-1][1], e)
            else:
                merged.append([b, e])
        parts = self.bgzf.read_ranges([(b, e) for b, e in merged])
        for (vb, _), p in zip(merged, parts):
            if p.shape[0] and p[-1] != 10:
                raise ValueError("%s: the index chunk at virtual offset %d does not end on a line boundary" % (self.path, vb))
        starts = np.cumsum([0] + [p.shape[0] for p in parts])
        buf = np.concatenate(parts) if parts else np.zeros(0, dtype=np.uint8)

        def where(off: int):
            k = int(np.searchsorted(starts, off, side="right")) - 1
            return "%s, line at virtual offset %d + %d bytes" % (self.path, merged[k][0], off - int(starts[k]))
        return buf, where

    def query(self, contig: str, beg: int, end: int) -> np.ndarray:
        """Fixed fields of the records overlapping [beg, end) of contig, in file order (host decode)."""
        tid = self.tids.get(contig)
        if tid is None:
            return np.zeros(0, dtype=L.VCF_REC_DTYPE)
        buf, where = self.fetch_union([(tid, beg, end)])
        recs = _lines(HostDecoder(), buf, where)
        keep = (_chrom_ids(buf, recs, self.tids, where) == tid) & (recs["pos0"] < end) & (recs["rend"] > beg)
        return recs[keep]


def _lines(dec, buf: np.ndarray, where) -> np.ndarray:
    recs = dec.lines(buf)
    bad = np.flatnonzero(recs["flags"] & L.VCF_BAD)
    if bad.shape[0]:
        off = int(recs["line_off"][bad[0]])
        line = buf[off: off + 60].tobytes().split(b"\n")[0]
        raise ValueError("%s: malformed VCF record %r (fewer than 8 columns, or POS / END not a valid position)"
                         % (where(off), line))
    return recs


def _chrom_ids(buf: np.ndarray, recs: np.ndarray, tids: Dict[str, int], where) -> np.ndarray:
    """Reference id of every line's CHROM (-1: not in the index), from the CHROM hashes; every line of a hash is
    checked byte for byte against the first."""
    out = np.full(recs.shape[0], -1, dtype=np.int64)
    if not recs.shape[0]:
        return out
    uh, inv = np.unique(recs["chrom_hash"], return_inverse=True)
    for g in range(uh.shape[0]):
        ix = np.flatnonzero(inv == g)
        ln = recs["chrom_len"][ix]
        off = recs["line_off"][ix]
        l0 = int(ln[0])
        name = buf[int(off[0]): int(off[0]) + l0].tobytes()
        same = ln == l0
        if l0 and same.all():
            same = (buf[off[:, None] + np.arange(l0)] == np.frombuffer(name, np.uint8)).all(axis=1)
        if not same.all():                       # a hash shared by two names: resolve this group one line at a time
            for i in ix.tolist():
                o, n = int(recs["line_off"][i]), int(recs["chrom_len"][i])
                out[i] = tids.get(buf[o:o + n].tobytes().decode("ascii", "replace"), -1)
            continue
        out[ix] = tids.get(name.decode("ascii", "replace"), -1)
    return out


# ------------------------------------------------------------------------------------------------
# site reader
# ------------------------------------------------------------------------------------------------

def query_plan(regions: Dict[str, List[Tuple[int, int]]], tids: Dict[str, int]):
    """Every merged interval of every contig, as ``pack_sites`` queries it -- [max(a, 0), max(b, 1)) by overlap: a list
    of (contig, reference id or None, intervals), and the (tid, beg, end) queries of the contigs the file has."""
    plan = [(contig, tids.get(contig), [(max(a, 0), max(b, 1)) for a, b in _merge(ivs)]) for contig, ivs in regions.items()]
    return plan, [(tid, beg, end) for _c, tid, iv in plan if tid is not None for beg, end in iv]


def select_records(plan, tid_of: np.ndarray, pos0: np.ndarray, rend: np.ndarray):
    """The records a region query per merged interval returns, in the order ``pack_sites`` visits them: (record indices,
    contig index of each into ``contigs``, ``contigs``).  ``tid_of`` / ``pos0`` / ``rend``: reference id, 0-based start
    and end of every decoded record (file order, so sorted by position within a reference).  A record that an earlier
    disjoint interval of its contig already returned is not returned again."""
    parts, cid_parts, contigs = [], [], []
    for contig, tid, iv in plan:
        if tid is None:
            continue
        ix_t = np.flatnonzero(tid_of == tid)                   # file order = sorted by position
        if not ix_t.shape[0]:
            continue
        pos_t = pos0[ix_t]
        span = int((rend[ix_t] - pos_t).max())
        prev_end = None
        got = []
        for beg, end in iv:
            lo = int(np.searchsorted(pos_t, beg - span, side="left"))
            hi = int(np.searchsorted(pos_t, end, side="left"))
            ix = ix_t[lo:hi]
            keep = rend[ix] > beg
            if prev_end is not None:
                # a record that starts before the end of the previous (disjoint) interval came back there already
                keep &= pos0[ix] >= prev_end
            got.append(ix[keep])
            prev_end = end
        sel_c = np.concatenate(got)
        if sel_c.shape[0]:
            parts.append(sel_c)
            cid_parts.append(np.full(sel_c.shape[0], len(contigs), dtype=np.int64))
            contigs.append(contig)
    sel = np.concatenate(parts) if parts else np.zeros(0, dtype=np.int64)
    cid = np.concatenate(cid_parts) if cid_parts else np.zeros(0, dtype=np.int64)
    return sel, cid, contigs


def member_columns(samples: Sequence[str], trios: Sequence[Tuple[str, str, str]]):
    """The member columns of the trios whose three samples are all in the file: (slot_of: sample -> column or -1, the
    number of columns, [(trio index, [column of kid, dad, mom])])."""
    sidx = {s: i for i, s in enumerate(samples)}
    cols_s = [(t, [sidx[m] for m in trio]) for t, trio in enumerate(trios) if all(m in sidx for m in trio)]
    slot_of = np.full(len(samples), -1, dtype=np.int32)
    n_members = 0
    for _t, ix in cols_s:
        for s in ix:
            if slot_of[s] < 0:
                slot_of[s] = n_members
                n_members += 1
    return slot_of, n_members, [(t, [int(slot_of[s]) for s in ix]) for t, ix in cols_s]


def read_sites(path, trios: Sequence[Tuple[str, str, str]], regions: Dict[str, List[Tuple[int, int]]], engine=None,
               max_digits: int = FAST_DIGITS) -> SiteTable:
    """``packers.pack_sites(VCF(path), trios, regions)`` from the file directly.  ``path``: a file name or a
    ``VcfFile``.  With ``engine`` the text is decoded on that engine's GPU (``Engine.vcf_decoder``).  ``max_digits``:
    significant digits a float GQ may have to be decoded natively (0 sends every float GQ to the host decode)."""
    vf = path if isinstance(path, VcfFile) else VcfFile(path)
    slot_of, n_members, cols = member_columns(vf.samples, trios)
    plan, queries = query_plan(regions, vf.tids)
    buf, where = vf.fetch_union(queries)
    dec = engine.vcf_decoder() if engine is not None else HostDecoder()
    recs = _lines(dec, buf, where)
    tid_of = _chrom_ids(buf, recs, vf.tids, where)
    pos0 = recs["pos0"].astype(np.int64)
    rend = recs["rend"].astype(np.int64)
    sel, cid, contigs = select_records(plan, tid_of, pos0, rend)
    r = recs[sel]
    simple = (r["flags"] & L.VCF_SIMPLE) != 0
    alt_b = np.zeros(sel.shape[0], dtype=np.uint8)
    has_alt = (r["n_alt"] > 0) & (r["alt_len"] > 0)
    alt_b[has_alt] = buf[(r["line_off"] + r["alt_off"])[has_alt]]
    refalt = {}
    for i in np.flatnonzero(~simple).tolist():
        o = int(r["line_off"][i])
        ref = buf[o + int(r["ref_off"][i]): o + int(r["ref_off"][i]) + int(r["ref_len"][i])].tobytes().decode()
        alt = buf[o + int(r["alt_off"][i]): o + int(r["alt_off"][i]) + int(r["alt_len"][i])].tobytes().decode()
        refalt[i] = (ref, [] if alt == "." else alt.split(","))
    cells = dec.samples(sel, slot_of, n_members, vf.gq_float(), max_digits)
    finish_cells(cells, buf, recs, sel, where)
    return build_site_table(trios, cols, contigs, cid, pos0[sel], simple, r["ref0"].astype(np.uint8), alt_b,
                            cells["gt"], cells["gq"], cells["rd"], cells["ad"], refalt)


# ------------------------------------------------------------------------------------------------
# DNM reader
# ------------------------------------------------------------------------------------------------

def read_dnms(path: str):
    """The DNMs of a plain or gzip / bgzip-compressed VCF, read whole without an index: for every record and every
    sample whose genotype is HET or HOM_ALT, in header order, {chrom, start, end, kid, vartype, bam: ""} with start the
    0-based POS, end tabix's end (INFO END, else start + len(REF)) and vartype INFO SVTYPE or "POINT" -- what
    ``unfazed.read_vars_vcf`` yields from cyvcf2."""
    from .utils import SNV_TYPES
    opener = gzip.open if path.endswith((".gz", ".bgz")) else open
    with opener(path, "rb") as f:
        data = f.read()
    if data and not data.endswith(b"\n"):
        data += b"\n"
    got = _parse_header(data, path)
    if got is None:
        raise ValueError("%s: no #CHROM header line" % path)
    samples, types, _chrom, body, _ = got
    buf = np.frombuffer(data, dtype=np.uint8)[body:]
    where = lambda off: "%s, line at byte %d" % (path, body + off)
    dec = HostDecoder()
    recs = _lines(dec, buf, where)
    sel = np.arange(recs.shape[0], dtype=np.int64)
    cells = dec.samples(sel, np.arange(len(samples), dtype=np.int32), len(samples),
                        types.get("GQ", "Float") != "Integer")
    finish_cells(cells, buf, recs, sel, where)
    gt = cells["gt"]
    for i in range(recs.shape[0]):
        o = int(recs["line_off"][i])
        cols = buf[o: o + int(recs["line_len"][i])].tobytes().decode().split("\t", 8)
        info = {}
        for kv in cols[7].split(";"):
            k, _, v = kv.partition("=")
            info.setdefault(k, v)
        vartype = info.get("SVTYPE") or SNV_TYPES[0]
        for s in np.flatnonzero((gt[i] == HET) | (gt[i] == HOM_ALT)).tolist():
            yield {"chrom": cols[0], "start": int(recs["pos0"][i]), "end": int(recs["rend"][i]), "kid": samples[s],
                   "vartype": vartype, "bam": ""}


# ------------------------------------------------------------------------------------------------
# phased VCF writer
# ------------------------------------------------------------------------------------------------

UNFAZED_LINE = ("##unfazed=%s. Phase info in pipe-separated GT field order -> 1|0 is paternal, 0|1 is maternal")
UOPS_LINE = ('##FORMAT=<ID=UOPS,Number=1,Type=Float,Description="Count of pieces of evidence supporting the '
             'unfazed-identified origin parent or `-1` if missing">')
UET_LINE = ('##FORMAT=<ID=UET,Number=1,Type=Float,Description="Unfazed evidence type: `0` (readbacked), `1` '
            '(allele-balance, for CNVs only), `2` (both), `3` (ambiguous readbacked), `4` (ambiguous allele-balance), '
            '`5` (ambiguous both), `6` (auto-phased sex-chromosome variant in male), or `-1` (missing)">')
PASS_LINE = '##FILTER=<ID=PASS,Description="All filters passed">'
_ID_RE = re.compile(rb"^##(FORMAT|FILTER)=<ID=([^,>]+)[,>]")


def phased_header(head: bytes, version: str) -> bytes:
    """The header of the phased VCF: the input's lines verbatim (a trailing '\\r' dropped), the PASS filter after
    ``##fileformat`` when the input declares none (htslib's header parser adds it), and before ``#CHROM`` the
    ``##unfazed=`` line and the UOPS / UET FORMAT lines not already declared."""
    lines = [x[:-1] if x.endswith(b"\r") else x for x in head.split(b"\n")]
    if lines and lines[-1] == b"":
        lines.pop()
    ids = {(m.group(1), m.group(2)) for m in map(_ID_RE.match, lines) if m}
    out = []
    for x in lines:
        if x.startswith(b"#CHROM"):
            out.append((UNFAZED_LINE % version).encode())
            for key, line in ((b"UOPS", UOPS_LINE), (b"UET", UET_LINE)):
                if (b"FORMAT", key) not in ids:
                    out.append(line.encode())
        out.append(x)
    if (b"FILTER", b"PASS") not in ids:
        at = 1 if out and out[0].startswith(b"##fileformat") else 0
        out.insert(at, PASS_LINE.encode())
    return b"\n".join(out) + b"\n"


def _svtype(buf: np.ndarray, rec) -> str:
    """INFO SVTYPE of a line as ``read_dnms`` takes it (the first SVTYPE key; "POINT" when absent or empty)."""
    from .utils import SNV_TYPES
    o = int(rec["line_off"])
    cols = buf[o: o + int(rec["line_len"])].tobytes().decode().split("\t", 8)
    for kv in cols[7].split(";"):
        k, _, v = kv.partition("=")
        if k == "SVTYPE":
            return v or SNV_TYPES[0]
    return SNV_TYPES[0]


def match_edits(pos0: np.ndarray, rend: np.ndarray, chrom_of, svtype_of, kid_gts, samples: Sequence[str], read_records,
                include_ambiguous, verbose, evidence_min_ratio):
    """The edit list of the phased cells of a DNM list's records (``_lib.VCF_EDIT_DTYPE`` sorted by (record, sample),
    and its CSR offsets by record), in O(#records); the core of both phased writers (``phase_edits`` here, and
    ``bcfio.phase_edits``).  The candidate records are those whose (CHROM, pos0, end) is some phasing record's region;
    their genotypes are decoded for the kids only, and every HET / HOM_ALT cell whose key
    ``{CHROM}_{pos0}_{end}_{sample}_{SVTYPE or POINT}`` is a phasing record gets that record's call.  ``chrom_of(i)`` /
    ``svtype_of(i)``: CHROM and SVTYPE (or "POINT") of record i; ``kid_gts(sel, kids)``: the genotype codes
    [len(sel), len(kids)] of the samples ``kids`` in the records ``sel``."""
    from .unfazed import summarize_record, uet_code
    n = int(pos0.shape[0])
    regions = {(str(r["region"]["chrom"]), int(r["region"]["start"]), int(r["region"]["end"]))
               for r in read_records.values()}
    sidx = {s: i for i, s in enumerate(samples)}
    kids = sorted({sidx[r["kid"]] for r in read_records.values() if r.get("kid") in sidx})
    rows = []
    if regions and kids and n:
        pe = np.array(sorted({(p, e) for _c, p, e in regions}), dtype=np.int64)
        key_l = pos0.astype(np.int64) * (1 << 32) + rend.astype(np.int64)
        cand = np.flatnonzero(np.isin(key_l, pe[:, 0] * (1 << 32) + pe[:, 1]))
        chrom = {}
        keep = []
        for i in cand.tolist():
            c = chrom_of(i)
            if (c, int(pos0[i]), int(rend[i])) in regions:
                chrom[i] = c
                keep.append(i)
        if keep:
            gt = kid_gts(np.array(keep, dtype=np.int64), kids)
            for li, i in enumerate(keep):
                carriers = np.flatnonzero((gt[li] == HET) | (gt[li] == HOM_ALT))
                if not carriers.shape[0]:
                    continue
                head = "%s_%d_%d_" % (chrom[i], int(pos0[i]), int(rend[i]))
                tail = "_" + svtype_of(i)
                for m in carriers.tolist():
                    key = head + samples[kids[m]] + tail
                    rec = read_records.get(key)
                    if rec is None:
                        continue
                    s = summarize_record(rec, include_ambiguous, verbose, evidence_min_ratio)
                    if s is None:
                        continue
                    phase = 1 if s["origin_parent"] == rec["dad"] else 2 if s["origin_parent"] == rec["mom"] else 0
                    rows.append((i, kids[m], phase, int(s["evidence_count"]), uet_code(s["evidence_types"])))
    rows.sort()
    edits = np.zeros(len(rows), dtype=L.VCF_EDIT_DTYPE)
    line = np.array([r[0] for r in rows], dtype=np.int64)
    for k, name in enumerate(("sample", "phase", "uops", "uet")):
        edits[name] = [r[k + 1] for r in rows]
    edit_off = np.searchsorted(line, np.arange(n + 1), side="left").astype(np.int64)
    return edit_off, edits


def phase_edits(buf: np.ndarray, recs: np.ndarray, samples: Sequence[str], read_records, include_ambiguous, verbose,
                evidence_min_ratio, dec=None):
    """``match_edits`` of the lines of a text DNM list: CHROM and SVTYPE from the text, the kids' genotypes from the
    decoder's ``samples``."""
    dec = dec or HostDecoder()

    def chrom_of(i):
        o = int(recs["line_off"][i])
        return buf[o: o + int(recs["chrom_len"][i])].tobytes().decode()

    def kid_gts(sel, kids):
        slot_of = np.full(len(samples), -1, dtype=np.int32)
        slot_of[kids] = np.arange(len(kids), dtype=np.int32)
        return dec.samples(sel, slot_of, len(kids), True)["gt"]
    return match_edits(recs["pos0"], recs["rend"], chrom_of, lambda i: _svtype(buf, recs[i]), kid_gts, samples,
                       read_records, include_ambiguous, verbose, evidence_min_ratio)


def write_output(outfile: str, head: bytes, body) -> None:
    """The header and body of a phased VCF to ``/dev/stdout``, to BGZF with an EOF block when ``outfile`` ends in
    ``.gz``, else to a plain file."""
    if outfile == "/dev/stdout":
        import sys
        sys.stdout.flush()
        sys.stdout.buffer.write(head)
        sys.stdout.buffer.write(memoryview(body))
        sys.stdout.buffer.flush()
    elif outfile.endswith(".gz"):
        write_bgzf(outfile, head, memoryview(body))
    else:
        with open(outfile, "wb") as f:
            f.write(head)
            f.write(memoryview(body))


def write_phased_vcf(in_path: str, read_records, include_ambiguous, verbose, outfile: str, evidence_min_ratio,
                     engine=None) -> None:
    """The phased VCF of ``unfazed.write_vcf_output`` without cyvcf2: every line of the plain or gzipped DNM VCF
    ``in_path`` with GT 1|0 (paternal) / 0|1 (maternal) and UOPS / UET for the phased carriers, UOPS = UET = -1 in
    every other cell.  The edit list is built on the host (``phase_edits``); the sample columns are rewritten in
    native code (csrc/vcfout.cu), on ``engine``'s GPU when given.  Bytes the contract does not touch are copied
    verbatim (DESIGN §5).  ``outfile``: ``/dev/stdout`` or a plain file, BGZF when it ends in ``.gz``."""
    from . import __version__
    opener = gzip.open if in_path.endswith((".gz", ".bgz")) else open
    with opener(in_path, "rb") as f:
        data = bytearray().join(iter(lambda: f.read(1 << 24), b""))      # writable: the device upload wraps it
    if data and not data.endswith(b"\n"):
        data += b"\n"
    got = _parse_header(data, in_path)
    if got is None:
        raise ValueError("%s: no #CHROM header line" % in_path)
    samples, _types, _chrom, body, _ = got
    buf = np.frombuffer(data, dtype=np.uint8)[body:]
    head_lines = data[:body].count(b"\n")
    where = lambda off: "%s, line %d" % (in_path, head_lines + 1 + int(np.searchsorted(ends, off, side="left")))
    dec = engine.vcf_decoder() if engine is not None else HostDecoder()
    recs = _lines(dec, buf, lambda off: "%s, line at byte %d" % (in_path, body + off))
    ends = (recs["line_off"] + recs["line_len"]).astype(np.int64)
    edit_off, edits = phase_edits(buf, recs, samples, read_records, include_ambiguous, verbose, evidence_min_ratio, dec)
    out, line_bad = dec.rewrite(edit_off, edits, len(samples))
    bad = np.flatnonzero(line_bad)
    if bad.shape[0]:
        i = int(bad[0])
        off = int(recs["line_off"][i])
        st = int(line_bad[i])
        if st & L.VCFOUT_COLUMNS:
            raise ValueError("%s: more sample columns than header samples" % where(off))
        if st & L.VCFOUT_FIELDS:
            raise ValueError("%s: a sample with more subfields than FORMAT keys" % where(off))
        cols = buf[off: off + int(recs["line_len"][i])].tobytes().decode("ascii", "replace").split("\t")
        gi = cols[8].split(":").index("GT")
        e = edits[int(edit_off[i]): int(edit_off[i + 1])]
        for s in e["sample"][e["phase"] != 0].tolist():
            sub = (cols[9 + s] if 9 + s < len(cols) else ".").split(":")
            gt = sub[gi] if gi < len(sub) else "."
            if "/" not in gt and "|" not in gt:
                raise ValueError("%s: the haploid GT %r of sample %s cannot be phased" % (where(off), gt, samples[s]))
    write_output(outfile, phased_header(data[:body], __version__), out)


# ------------------------------------------------------------------------------------------------
# writer
# ------------------------------------------------------------------------------------------------

_GT_TEXT = {HOM_REF: "0/0", HET: "0/1", HOM_ALT: "1/1", GT_UNKNOWN: "./."}


def _float_text(x: np.float32) -> str:
    return np.format_float_positional(x, unique=True, trim="-")


def write_vcf(table: SiteTable, path: str, end: Optional[Dict[int, int]] = None,
              format_order: Optional[Sequence[Sequence[str]]] = None, level: int = 6, index: str = "tbi",
              min_shift: int = 14, depth: Optional[int] = None) -> None:
    """Sorted ``path`` (.vcf.gz) + ``path.tbi`` (or with ``index="csi"`` ``path.csi`` of ``min_shift`` / ``depth``, depth
    None: the smallest that spans the records) of ``table``: one line per record (rows grouped by ``rec_id`` and contig,
    as ``oracle.fakes`` groups them into records), every sample of every trio, ``./.`` for a trio without a row in the
    record.  FORMAT GT:AD:GQ; GQ is declared Float when a value is not integral (written in the shortest text that
    parses back to the same float32) and Integer otherwise; AD is ``rd,ad`` (``.`` for -1).  ``end``: record index ->
    INFO END (1-based inclusive); ``format_order``: record index -> the order of GT / AD / GQ on that line."""
    t = table
    view_rows, g_lo, g_contig = _records(t)
    n_rec = g_lo.shape[0] - 1
    samples: List[str] = []
    for trio in t.trios:
        for s in trio:
            if s not in samples:
                samples.append(s)
    sidx = {s: i for i, s in enumerate(samples)}
    blk = np.repeat(np.arange(t.n_blocks), np.diff(t.blk_off))
    gq = t.gq
    is_float = bool(np.any((gq != np.round(gq)) & (gq != -1)))
    text_gq = np.empty(gq.shape, dtype=object)
    for m in range(3):
        if is_float:
            text_gq[m] = [_float_text(x) for x in gq[m]]
        else:
            text_gq[m] = [str(int(x)) for x in gq[m]]
        text_gq[m][gq[m] == -1] = "."
    if is_float:
        back = np.array([np.float32(float(x)) if x != "." else np.float32(-1) for x in text_gq.reshape(-1)],
                        dtype=np.float32).reshape(gq.shape)
        assert np.array_equal(back, gq), "GQ text does not parse back to the same float32"
    head = ["##fileformat=VCFv4.2"]
    for c in t.contigs:
        head.append("##contig=<ID=%s>" % c)
    head += ['##INFO=<ID=END,Number=1,Type=Integer,Description="End position">',
             '##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype">',
             '##FORMAT=<ID=AD,Number=R,Type=Integer,Description="Allelic depths">',
             '##FORMAT=<ID=GQ,Number=1,Type=%s,Description="Genotype quality">' % ("Float" if is_float else "Integer"),
             "\t".join(["#CHROM", "POS", "ID", "REF", "ALT", "QUAL", "FILTER", "INFO", "FORMAT"] + samples)]
    head_b = ("\n".join(head) + "\n").encode()
    dep = lambda v: "." if v == -1 else str(int(v))
    lines: List[bytes] = []
    pos0 = np.zeros(n_rec, dtype=np.int64)
    rend = np.zeros(n_rec, dtype=np.int64)
    fill: Dict[Tuple[str, ...], str] = {}
    for g in range(n_rec):
        rows = view_rows[g_lo[g]: g_lo[g + 1]]
        lead = int(rows[0])
        ref, alts = t.ref_alts(lead)
        p0 = int(t.pos[lead])
        order = tuple(format_order[g]) if format_order is not None else ("GT", "AD", "GQ")
        miss = "./." if order[0] == "GT" else ":".join("./." if k == "GT" else "." for k in order)
        cells = {}
        for row in rows.tolist():
            b = 3 * int(t.blk_trio[blk[row]])
            for m in range(3):
                v = {"GT": _GT_TEXT[int(t.gt[m, row])], "AD": "%s,%s" % (dep(t.rd[m, row]), dep(t.ad[m, row]))
                     if not (t.rd[m, row] == -1 and t.ad[m, row] == -1) else ".", "GQ": text_gq[m, row]}
                cells[sidx[t.trios[int(t.blk_trio[blk[row]])][m]]] = ":".join(v[k] for k in order)
        out, at = [], 0
        for s in sorted(cells):
            if s > at:
                out.append(_fill(fill, miss, s - at))
            out.append(cells[s])
            at = s + 1
        if at < len(samples):
            out.append(_fill(fill, miss, len(samples) - at))
        e = (end or {}).get(g)
        info = "END=%d" % e if e is not None else "."
        lines.append(("%s\t%d\t.\t%s\t%s\t.\tPASS\t%s\t%s\t%s\n" % (
            t.contigs[int(g_contig[g])], p0 + 1, ref, ",".join(alts) if alts else ".", info, ":".join(order),
            "\t".join(out))).encode())
        pos0[g] = p0
        rend[g] = e if (e is not None and e > p0) else p0 + len(ref)
    body = b"".join(lines)
    starts = np.cumsum([0] + [len(x) for x in lines]).astype(np.int64)
    voff = write_bgzf(path, head_b, body, level)
    names = b"".join(c.encode() + b"\0" for c in t.contigs)
    cols = (len(t.contigs), g_contig.astype(np.int64), pos0, rend, voff(starts[:-1]), voff(starts[1:]))
    if index == "csi":
        aux = struct.pack("<7i", 2, 1, 2, 0, ord("#"), 0, len(names)) + names
        write_csi(path + ".csi", *cols, min_shift=min_shift, depth=depth, aux=aux, level=level)
    elif index == "tbi":
        tbi = b"TBI\x01" + struct.pack("<8i", len(t.contigs), 2, 1, 2, 0, ord("#"), 0, len(names)) + names + index_refs(*cols)
        write_bgzf(path + ".tbi", tbi, b"", level)
    else:
        raise ValueError("index must be 'tbi' or 'csi', not %r" % index)


def _fill(cache: Dict, miss: str, k: int) -> str:
    key = (miss, k)
    s = cache.get(key)
    if s is None:
        s = cache[key] = "\t".join([miss] * k)
    return s


def _records(t: SiteTable):
    """Rows grouped into records as ``oracle.fakes._VcfView`` groups them: (rows in record order, group bounds,
    contig of each group)."""
    V = t.n_rows
    blk = np.repeat(np.arange(t.n_blocks), np.diff(t.blk_off))
    contig = t.blk_contig[blk].astype(np.int64)
    rid = t.record_ids().astype(np.int64)
    order = np.lexsort((blk, rid, t.pos.astype(np.int64), contig))
    srid = rid[order]
    first = np.ones(V, dtype=bool)
    first[1:] = (srid[1:] != srid[:-1]) | (contig[order][1:] != contig[order][:-1])
    g_first = np.flatnonzero(first)
    return order, np.concatenate([g_first, [V]]).astype(np.int64), contig[order][g_first]
