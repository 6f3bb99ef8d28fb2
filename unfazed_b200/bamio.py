"""Indexed BAM files without pysam: BGZF inflate and BAI region queries on the host, record decoding in native code.

* ``BamFile`` -- one coordinate-sorted BAM and its ``.bai`` (or ``.csi``): the header (reference names and lengths), the BAI bins,
  chunks and linear index, and region queries that return the records overlapping an interval (htslib's ``reg2bins``
  and linear-index minimum offset, ``bam_endpos`` overlap).  BGZF blocks are inflated with zlib in a thread pool
  (zlib releases the GIL), CRC32 and ISIZE checked, and cached by file offset for the length of one load.
* ``read_regions`` -- the ``ReadTable`` ``packers.pack_reads`` builds from pysam handles over the same reads, array
  for array.  Record boundaries, fixed fields and byte gathers are native (csrc/bam.cu, host functions); everything
  else is numpy over the inflated buffer -- no Python work per record except splitting the read names into a list.
  With ``engine=`` the bulk columns (CIGAR, bases, qualities) are decoded on the GPU instead and the table comes back
  as the host half of a device-decoded ``DeviceReads`` (``Engine.decode_bam``).
* ``write_bam`` -- a coordinate-sorted BAM + BAI or CSI from a ``ReadTable`` (tests and tools generate their inputs
  with it).
* ``CsiIndex`` / ``write_csi`` -- the CSI index (any ``min_shift`` / ``depth``) with the ``chunks`` queries of
  ``BaiIndex``; a BAM may come with a ``.csi`` instead of a ``.bai``, and ``vcfio`` and ``bcfio`` use it too.

CRAM is not read here; ``datasource.load_reads`` sends it to pysam.
"""
from __future__ import annotations

import ctypes as C
import mmap
import os
import struct
import zlib
from concurrent.futures import ThreadPoolExecutor
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import _lib as L
from .packers import _merge, _mate_join
from .schema import AUX_HAS_SA, AUX_SAME_REF, QUAL_ESCAPE, READ_HDR, ReadTable, pack_seq

BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
_BLOCK_IN = 0xFF00                       # uncompressed bytes per written block (htslib's BGZF_BLOCK_SIZE)
_THREADS = min(32, os.cpu_count() or 4)

# BAM base nibble (=ACMGRSVTWYHKDBN) -> 2-bit code / escape bit, as packers._BASE_LUT / _ESC_LUT map the letters
_NIB_CHARS = b"=ACMGRSVTWYHKDBN"
_NIB_CODE = np.array([1, 0, 1, 1, 2, 1, 1, 1, 3, 1, 1, 1, 1, 1, 1, 0], dtype=np.uint8)
_NIB_ESC = np.array([c not in b"ACGT" for c in _NIB_CHARS], dtype=bool)
_FIXED = np.dtype([("block_size", "<i4"), ("ref_id", "<i4"), ("pos", "<i4"), ("l_name", "u1"), ("mapq", "u1"),
                   ("bin", "<u2"), ("n_cigar", "<u2"), ("flag", "<u2"), ("l_seq", "<i4"), ("next_ref_id", "<i4"),
                   ("next_pos", "<i4"), ("tlen", "<i4")])
assert _FIXED.itemsize == 36


def _ptr(a: np.ndarray) -> int:
    return a.ctypes.data


def _lib():
    return L.load()


# ------------------------------------------------------------------------------------------------
# native helpers (host functions of libunfazed_sm100.so)
# ------------------------------------------------------------------------------------------------

def record_offsets(buf: np.ndarray, max_records: Optional[int] = None) -> Tuple[np.ndarray, int]:
    """Byte offsets of the records of ``buf`` (walking block_size from 0) and where the walk stopped."""
    n = int(buf.shape[0])
    cap = n // 36 + 1 if max_records is None else min(int(max_records), n // 36 + 1)
    offs = np.empty(cap, dtype=np.int64)
    end = C.c_int64(0)
    got = _lib().unfz_bam_record_offsets(_ptr(buf), n, cap, _ptr(offs), C.byref(end))
    if got < 0:
        raise ValueError("malformed BAM record at byte %d of the inflated data (block_size < 32)" % end.value)
    return offs[:got], int(end.value)


def parse_records(buf: np.ndarray, offs: np.ndarray) -> np.ndarray:
    """Fixed fields of the records at ``offs`` (``_lib.BAM_REC_DTYPE``); the same code as the device parse."""
    offs = np.ascontiguousarray(offs, dtype=np.int64)
    out = np.empty(offs.shape[0], dtype=L.BAM_REC_DTYPE)
    bad = _lib().unfz_bam_parse_host(_ptr(buf), int(buf.shape[0]), _ptr(offs), int(offs.shape[0]), _ptr(out))
    if bad:
        raise ValueError("%d malformed BAM record(s): fields or aux tags overrun block_size" % bad)
    return out


def gather(buf: np.ndarray, src: np.ndarray, length: np.ndarray) -> np.ndarray:
    """The byte ranges [src[i], src[i] + length[i]) of ``buf``, back to back."""
    src = np.ascontiguousarray(src, dtype=np.int64)
    length = np.ascontiguousarray(length, dtype=np.int64)
    out = np.empty(int(length.sum()), dtype=np.uint8)
    if out.shape[0]:
        _lib().unfz_bam_gather_host(_ptr(buf), _ptr(src), _ptr(length), int(src.shape[0]), _ptr(out))
    return out


# ------------------------------------------------------------------------------------------------
# BGZF
# ------------------------------------------------------------------------------------------------

class BgzfReader:
    """Random access to the BGZF blocks of one file.  Inflated blocks are cached by file offset (one load)."""

    def __init__(self, path: str):
        self.path = path
        with open(path, "rb") as f:
            size = os.fstat(f.fileno()).st_size
            self.data = mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ) if size else b""
        if len(self.data) < len(BGZF_EOF) or self.data[len(self.data) - len(BGZF_EOF):] != BGZF_EOF:
            raise ValueError("%s: no BGZF EOF block at the end (truncated file?)" % path)
        self._size: Dict[int, int] = {}          # compressed block size by offset
        self._cache: Dict[int, bytes] = {}

    def block_size(self, coff: int) -> int:
        s = self._size.get(coff)
        if s is None:
            d = self.data
            if coff + 18 > len(d):
                raise ValueError("%s: truncated BGZF block header at offset %d" % (self.path, coff))
            if d[coff:coff + 4] != b"\x1f\x8b\x08\x04":
                raise ValueError("%s: no BGZF block at offset %d" % (self.path, coff))
            xlen = struct.unpack_from("<H", d, coff + 10)[0]
            p, e, s = coff + 12, coff + 12 + xlen, None
            while p + 4 <= e:
                si1, si2, slen = d[p], d[p + 1], struct.unpack_from("<H", d, p + 2)[0]
                if si1 == 66 and si2 == 67 and slen == 2:
                    s = struct.unpack_from("<H", d, p + 4)[0] + 1
                p += 4 + slen
            if s is None:
                raise ValueError("%s: gzip member at offset %d has no BC (BSIZE) subfield" % (self.path, coff))
            if coff + s > len(d):
                raise ValueError("%s: truncated BGZF block at offset %d" % (self.path, coff))
            self._size[coff] = s
        return s

    def _inflate(self, coff: int) -> bytes:
        d = self.data
        s = self.block_size(coff)
        xlen = struct.unpack_from("<H", d, coff + 10)[0]
        raw = zlib.decompress(d[coff + 12 + xlen: coff + s - 8], -15)
        crc, isize = struct.unpack_from("<II", d, coff + s - 8)
        if len(raw) != isize or zlib.crc32(raw) != crc:
            raise ValueError("%s: BGZF block at offset %d fails its CRC32/ISIZE check" % (self.path, coff))
        return raw

    def inflate(self, coffs: Sequence[int]) -> List[bytes]:
        """Inflated blocks at these file offsets (uncached ones in the thread pool)."""
        todo = sorted({c for c in coffs if c not in self._cache})
        if len(todo) > 1:
            with ThreadPoolExecutor(_THREADS) as ex:
                for c, raw in zip(todo, ex.map(self._inflate, todo)):
                    self._cache[c] = raw
        elif todo:
            self._cache[todo[0]] = self._inflate(todo[0])
        return [self._cache[c] for c in coffs]

    def blocks_between(self, cbeg: int, cend: int) -> List[int]:
        """Offsets of the blocks from cbeg up to (excluding) cend."""
        out, c = [], cbeg
        while c < cend:
            out.append(c)
            c += self.block_size(c)
        return out

    def read_ranges(self, ranges: Sequence[Tuple[int, int]]) -> List[np.ndarray]:
        """Uncompressed bytes of virtual-offset ranges [vbeg, vend); all their blocks inflated together."""
        plans = []
        need: List[int] = []
        for vb, ve in ranges:
            cb, ub, ce, ue = vb >> 16, vb & 0xFFFF, ve >> 16, ve & 0xFFFF
            blocks = self.blocks_between(cb, ce) + ([ce] if ue else [])
            plans.append((blocks, ub, ue, ce))
            need += blocks
        self.inflate(need)
        out = []
        for blocks, ub, ue, ce in plans:
            parts = [self._cache[c] for c in blocks]
            joined = b"".join(parts)
            stop = len(joined) - (len(parts[-1]) - ue if (ue and blocks and blocks[-1] == ce) else 0)
            out.append(np.frombuffer(joined, dtype=np.uint8)[ub:stop])
        return out

    def stream_from(self, vbeg: int, min_bytes: int, step_blocks: int = 64):
        """Uncompressed bytes from vbeg on, at least ``min_bytes`` of them or up to the end of the file."""
        cb, ub = vbeg >> 16, vbeg & 0xFFFF
        blocks, c = [], cb
        eof = len(self.data) - len(BGZF_EOF)
        have = 0
        while c < eof:
            chunk = []
            while c < eof and len(chunk) < step_blocks:
                chunk.append(c)
                c += self.block_size(c)
            got = self.inflate(chunk)
            blocks += chunk
            have += sum(len(g) for g in got)
            if have - ub >= min_bytes:
                break
        joined = b"".join(self._cache[b] for b in blocks)
        return np.frombuffer(joined, dtype=np.uint8)[ub:], c >= eof


def _bgzf_block(raw: bytes, level: int) -> bytes:
    co = zlib.compressobj(level, zlib.DEFLATED, -15)
    cdata = co.compress(raw) + co.flush()
    bsize = 18 + len(cdata) + 8
    hdr = b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", bsize - 1)
    return hdr + cdata + struct.pack("<II", zlib.crc32(raw), len(raw))


# ------------------------------------------------------------------------------------------------
# BAI
# ------------------------------------------------------------------------------------------------

def reg2bins(beg: int, end: int, min_shift: int = 14, depth: int = 5) -> List[int]:
    """htslib's reg2bins: the bins that may hold records overlapping [beg, end) (0-based, half-open) in a binning of
    ``depth`` levels below the root whose leaves span 2^min_shift bases ((14, 5): BAI and TBI)."""
    if beg >= end:
        return []
    end -= 1
    bins: List[int] = []
    s, t = min_shift + 3 * depth, 0
    for lvl in range(depth + 1):
        bins += range(t + (beg >> s), t + (end >> s) + 1)
        s -= 3
        t += 1 << (3 * lvl)
    return bins


def reg2bin(beg: int, end: int, min_shift: int = 14, depth: int = 5) -> int:
    """htslib's reg2bin: the smallest bin containing [beg, end)."""
    end -= 1
    s, t = min_shift, ((1 << (3 * depth)) - 1) // 7
    for lvl in range(depth, 0, -1):
        if beg >> s == end >> s:
            return t + (beg >> s)
        s += 3
        t -= 1 << (3 * (lvl - 1))
    return 0


def bin_first(lvl: int) -> int:
    """The first bin of level ``lvl`` (the root is level 0)."""
    return ((1 << (3 * lvl)) - 1) // 7


def pseudo_bin(depth: int) -> int:
    """The bin number that holds the mapped / unmapped counts of a reference (37450 at depth 5)."""
    return bin_first(depth + 1) + 1


def parse_bins(d: bytes, p: int, n_ref: int) -> Tuple[List[Dict[int, np.ndarray]], List[np.ndarray], int]:
    """The per-reference part BAI and TBI share, from byte p of the index: bins (bin -> chunk array [n, 2] of virtual
    offsets, the pseudo-bin 37450 of counts dropped) and the linear index of every reference, and where it ended."""
    bins_all: List[Dict[int, np.ndarray]] = []
    linear: List[np.ndarray] = []
    for _ in range(n_ref):
        n_bin = struct.unpack_from("<i", d, p)[0]
        p += 4
        bins = {}
        for _ in range(n_bin):
            b, n_chunk = struct.unpack_from("<Ii", d, p)
            p += 8
            ch = np.frombuffer(d, dtype="<u8", count=2 * n_chunk, offset=p).reshape(n_chunk, 2)
            p += 16 * n_chunk
            if b != 37450:                    # pseudo-bin of mapped / unmapped counts
                bins[b] = ch
        n_intv = struct.unpack_from("<i", d, p)[0]
        p += 4
        linear.append(np.frombuffer(d, dtype="<u8", count=n_intv, offset=p).copy())
        p += 8 * n_intv
        bins_all.append(bins)
    return bins_all, linear, p


class BaiIndex:
    """Bins (bin -> chunk array [n, 2] of virtual offsets) and linear index of every reference."""
    min_shift, depth = 14, 5

    def __init__(self, path: str):
        d = open(path, "rb").read()
        if d[:4] != b"BAI\x01":
            raise ValueError("%s: not a BAI index" % path)
        n_ref = struct.unpack_from("<i", d, 4)[0]
        self.bins, self.linear, _ = parse_bins(d, 8, n_ref)

    def min_offset(self, tid: int, beg: int) -> int:
        """The virtual offset before which no record overlapping beg starts: the linear index at beg's 16 kb window."""
        lin = self.linear[tid]
        return int(lin[min(beg >> 14, lin.shape[0] - 1)]) if lin.shape[0] else 0

    def chunks(self, tid: int, beg: int, end: int) -> List[Tuple[int, int]]:
        """Merged chunk list of [beg, end) on reference tid: the chunks of reg2bins' bins that end after the minimum
        offset (``min_offset``), sorted and merged.  A zero-length interval asks for the records covering beg (the
        overlap test pos < end and bam_endpos > beg is the caller's)."""
        end = max(end, beg + 1)
        if tid < 0 or tid >= len(self.bins):
            return []
        bins = self.bins[tid]
        min_off = self.min_offset(tid, beg)
        ch = [bins[b] for b in reg2bins(beg, end, self.min_shift, self.depth) if b in bins]
        if not ch:
            return []
        c = np.concatenate(ch)
        c = c[c[:, 1] > min_off]
        if not c.shape[0]:
            return []
        c = c[np.argsort(c[:, 0], kind="stable")]
        out = [[int(c[0, 0]), int(c[0, 1])]]
        for b, e in c[1:].tolist():
            if b <= out[-1][1]:
                out[-1][1] = max(out[-1][1], e)
            else:
                out.append([b, e])
        return [(max(b, min_off), e) for b, e in out]


class CsiIndex(BaiIndex):
    """A CSI index (BGZF-compressed): ``min_shift`` and ``depth`` of its binning, the ``aux`` bytes (a tabix header for a
    .vcf.gz, empty for BCF and BAM; ``names`` holds the reference names of a tabix header, else None), and per
    reference the bins with their chunks and ``loffset``.  There is no linear index: the minimum offset of a query is the
    ``loffset`` of the nearest existing bin at or left of beg's leaf bin, walking towards the root (htslib's
    ``hts_itr_query``).  Region queries are ``BaiIndex.chunks``."""

    def __init__(self, path: str):
        raw, _ = BgzfReader(path).stream_from(0, 1 << 62)
        d = raw.tobytes()
        if d[:4] != b"CSI\x01" or len(d) < 16:
            raise ValueError("%s: not a CSI index" % path)
        self.min_shift, self.depth, l_aux = struct.unpack_from("<3i", d, 4)
        if not (0 < self.min_shift and 0 < self.depth and self.min_shift + 3 * self.depth < 64) or l_aux < 0:
            raise ValueError("%s: CSI min_shift %d / depth %d out of range" % (path, self.min_shift, self.depth))
        self.aux = d[16:16 + l_aux]
        self.names = None
        if l_aux >= 28:                                        # tabix header: format, columns, meta, skip, names
            l_nm = struct.unpack_from("<i", self.aux, 24)[0]
            self.names = [x.decode() for x in self.aux[28:28 + l_nm].split(b"\0") if x]
        p = 16 + l_aux
        try:
            n_ref = struct.unpack_from("<i", d, p)[0]
            p += 4
            pseudo = pseudo_bin(self.depth)
            self.bins, self.loff = [], []
            for _ in range(n_ref):
                n_bin = struct.unpack_from("<i", d, p)[0]
                p += 4
                bins, loff = {}, {}
                for _ in range(n_bin):
                    b, lo, n_chunk = struct.unpack_from("<IQi", d, p)
                    p += 16
                    ch = np.frombuffer(d, dtype="<u8", count=2 * n_chunk, offset=p).reshape(n_chunk, 2)
                    p += 16 * n_chunk
                    if b != pseudo:
                        bins[b], loff[b] = ch, lo
                self.bins.append(bins)
                self.loff.append(loff)
        except (struct.error, ValueError):
            raise ValueError("%s: truncated CSI index" % path)

    def min_offset(self, tid: int, beg: int) -> int:
        loff = self.loff[tid]
        b = bin_first(self.depth) + (beg >> self.min_shift)
        while b and b not in loff:
            first = (((b - 1) >> 3) << 3) + 1                  # the first child of b's parent
            b = b - 1 if b > first else (b - 1) >> 3
        return loff.get(b, 0)


def open_index(path: str):
    """The BAI (uncompressed, ``BAI\\1``) or CSI (BGZF) index of a BAM at ``path``, by its first bytes."""
    with open(path, "rb") as f:
        head = f.read(4)
    return BaiIndex(path) if head == b"BAI\x01" else CsiIndex(path)


# ------------------------------------------------------------------------------------------------
# BAM file
# ------------------------------------------------------------------------------------------------

def index_path(path: str) -> Optional[str]:
    """The index of a BAM: ``<file>.bam.bai`` or ``<file>.bai`` if one exists, else ``<file>.bam.csi`` or
    ``<file>.csi``."""
    stem = os.path.splitext(path)[0]
    for p in (path + ".bai", stem + ".bai", path + ".csi", stem + ".csi"):
        if os.path.exists(p):
            return p
    return None


class BamFile:
    """One indexed BAM: header, BAI or CSI index and region queries.  Records come back as (buffer, offsets, parsed
    fields)."""

    def __init__(self, path: str, index: Optional[str] = None):
        self.path = path
        self.bgzf = BgzfReader(path)
        ip = index or index_path(path)
        if ip is None:
            raise ValueError("%s: no .bai or .csi index" % path)
        self.bai = open_index(ip)
        head, _ = self.bgzf.stream_from(0, 1 << 16)
        hb = head.tobytes()
        need = 12
        while True:
            try:
                self._parse_header(hb)
                break
            except struct.error:
                need = len(hb) * 2
                head, eof = self.bgzf.stream_from(0, need)
                if len(head) <= len(hb):
                    raise ValueError("%s: truncated BAM header" % path)
                hb = head.tobytes()
        # virtual offset of the first record: the header's uncompressed length mapped onto the blocks
        u, c = self.header_bytes, 0
        eof = len(self.bgzf.data) - len(BGZF_EOF)
        while c < eof:
            n = len(self.bgzf.inflate([c])[0])
            if u < n:
                break
            u -= n
            c += self.bgzf.block_size(c)
        self.first_voff = (c << 16) | u

    def _parse_header(self, b: bytes):
        if b[:4] != b"BAM\x01":
            raise ValueError("%s: not a BAM file" % self.path)
        l_text = struct.unpack_from("<i", b, 4)[0]
        p = 8 + l_text
        self.text = b[8:p].split(b"\0", 1)[0].decode("ascii", "replace")
        n_ref = struct.unpack_from("<i", b, p)[0]
        p += 4
        names, lens = [], []
        for _ in range(n_ref):
            ln = struct.unpack_from("<i", b, p)[0]
            if p + 4 + ln + 4 > len(b):
                raise struct.error("short")
            names.append(b[p + 4: p + 4 + ln].rstrip(b"\0").decode())
            lens.append(struct.unpack_from("<i", b, p + 4 + ln)[0])
            p += 8 + ln
        self.refs, self.ref_lens = names, lens
        self.tids = {n: i for i, n in enumerate(names)}
        self.header_bytes = p

    def tid(self, contig: str) -> int:
        t = self.tids.get(contig)
        if t is None:
            raise ValueError("invalid contig `%s`" % contig)
        return t

    def fetch_records(self, queries: Sequence[Tuple[int, int, int]]) -> Tuple[np.ndarray, np.ndarray]:
        """Inflated bytes of the chunks of every (tid, beg, end) query, back to back, and the record offsets of each
        query's chunks (a list of arrays into the one buffer).  Selection is left to the caller (``overlap``)."""
        ranges, owner = [], []
        for qi, (tid, beg, end) in enumerate(queries):
            for r in self.bai.chunks(tid, beg, end):
                ranges.append(r)
                owner.append(qi)
        return self._read_chunks(ranges, owner, len(queries))

    def fetch_union(self, queries: Sequence[Tuple[int, int, int]]) -> Tuple[np.ndarray, np.ndarray]:
        """Inflated bytes and record offsets of the UNION of the chunk lists of many (tid, beg, end) queries: every
        chunk is read once however many queries share it."""
        ch = sorted(c for tid, beg, end in queries for c in self.bai.chunks(tid, beg, end))
        merged: List[List[int]] = []
        for b, e in ch:
            if merged and b <= merged[-1][1]:
                merged[-1][1] = max(merged[-1][1], e)
            else:
                merged.append([b, e])
        buf, (offs,) = self._read_chunks([(b, e) for b, e in merged], [0] * len(merged), 1)
        return buf, offs

    def _read_chunks(self, ranges, owner, n_out):
        parts = self.bgzf.read_ranges(ranges)
        offs: List[List[np.ndarray]] = [[] for _ in range(n_out)]
        base = 0
        for qi, part in zip(owner, parts):
            o, stop = record_offsets(part)
            if stop != part.shape[0]:
                raise ValueError("%s: a BAI chunk does not end on a record boundary" % self.path)
            offs[qi].append(o + base)
            base += part.shape[0]
        buf = np.concatenate(parts) if parts else np.zeros(0, dtype=np.uint8)
        return buf, [np.concatenate(o) if o else np.zeros(0, dtype=np.int64) for o in offs]

    def head_tlen(self, n: int) -> np.ndarray:
        """Template lengths of the first n records of the file."""
        if n <= 0:
            return np.zeros(0, dtype=np.int64)
        want = 400 * n
        while True:
            buf, eof = self.bgzf.stream_from(self.first_voff, want)
            offs, _ = record_offsets(buf, n)
            if offs.shape[0] >= n or eof:
                break
            want *= 4
        idx = offs[:, None] + np.arange(32, 36)
        return buf[idx].copy().view("<i4").reshape(-1).astype(np.int64)

    def query(self, contig: str, beg: int, end: int):
        """Records overlapping [beg, end) of contig (ValueError for an unknown contig), in file order:
        (buffer, offsets, parsed fields).  Overlap is htslib's: pos < end and bam_endpos > beg."""
        tid = self.tid(contig)
        buf, (offs,) = self.fetch_records([(tid, beg, end)])
        rec = parse_records(buf, offs)
        keep = (rec["ref_id"] == tid) & (rec["pos"] < end) & (rec["end"] > beg)
        return buf, offs[keep], rec[keep]


# ------------------------------------------------------------------------------------------------
# region reader
# ------------------------------------------------------------------------------------------------

class _Records:
    """Records gathered over one load: inflated buffers back to back, record offsets, parsed fields."""

    def __init__(self, parse):
        self.parse = parse
        self.bufs: List[np.ndarray] = []
        self.size = 0
        self.offs: List[np.ndarray] = []
        self.rec: List[np.ndarray] = []
        self.names: List[str] = []
        self.n = 0

    def add(self, buf: np.ndarray, offs_list: List[np.ndarray]) -> List[np.ndarray]:
        """Adds one buffer with several offset lists; returns the global record indices of each list."""
        cat = np.concatenate(offs_list) if offs_list else np.zeros(0, dtype=np.int64)
        rec = self.parse(buf, cat, len(self.bufs))
        self.names += _names(buf, cat, rec["l_name"])
        self.bufs.append(buf)
        self.offs.append(cat + self.size)
        self.rec.append(rec)
        self.size += int(buf.shape[0])
        out, i = [], self.n
        for o in offs_list:
            out.append(np.arange(i, i + o.shape[0], dtype=np.int64))
            i += o.shape[0]
        self.n = i
        return out

    def finish(self):
        self.all_offs = np.concatenate(self.offs) if self.offs else np.zeros(0, dtype=np.int64)
        self.all_rec = np.concatenate(self.rec) if self.rec else np.zeros(0, dtype=L.BAM_REC_DTYPE)

    def gather(self, src: np.ndarray, length: np.ndarray) -> np.ndarray:
        """``gather`` over the buffers back to back, without joining them (``src``: offsets in the joined space)."""
        src = np.asarray(src, dtype=np.int64)
        length = np.asarray(length, dtype=np.int64)
        out = np.empty(int(length.sum()), dtype=np.uint8)
        dst = np.cumsum(length) - length
        base = np.cumsum([0] + [b.shape[0] for b in self.bufs])
        part = np.searchsorted(base, src, side="right") - 1
        for p, b in enumerate(self.bufs):
            m = np.flatnonzero(part == p)
            if m.shape[0] == 0:
                continue
            piece = gather(b, src[m] - base[p], length[m])
            out[_ranges(dst[m], length[m])] = piece
        return out

    def buffer(self) -> np.ndarray:
        return np.concatenate(self.bufs) if self.bufs else np.zeros(0, dtype=np.uint8)


def resolve_left_mates(mate: np.ndarray, names: List[str], flag: np.ndarray, blk_off: np.ndarray) -> np.ndarray:
    """The reads the device join marks -2 (hash collision, or its own candidate) resolved by name as
    ``packers._mate_join`` resolves them: the first other read of the block with that name, the other segment bit and
    no secondary / supplementary bit, or -1."""
    left = np.flatnonzero(mate == -2)
    if left.shape[0]:
        blk = np.searchsorted(blk_off, left, side="right") - 1
        by_name: Dict[Tuple[int, str], List[int]] = {}
        for b in sorted(set(blk.tolist())):
            for c in range(int(blk_off[b]), int(blk_off[b + 1])):
                by_name.setdefault((b, names[c]), []).append(c)
        for i, b in zip(left.tolist(), blk.tolist()):
            want = 0x80 if int(flag[i]) & 0x40 else 0x40
            mate[i] = next((c for c in by_name[(b, names[i])] if c != i and (int(flag[c]) & want)
                            and not (int(flag[c]) & 0x900)), -1)
    return mate


def _names(buf: np.ndarray, offs: np.ndarray, l_name: np.ndarray) -> List[str]:
    if offs.shape[0] == 0:
        return []
    raw = gather(buf, offs + 36, l_name.astype(np.int64))
    return raw.tobytes().decode("ascii", "replace").split("\0")[:-1]


def read_regions(paths: Dict[str, str], regions: Dict[str, Dict[str, List[Tuple[int, int]]]], head_reads: int = 0,
                 engine=None, min_gt_qual=20) -> ReadTable:
    """Reads of every kid overlapping the requested regions, plus their mates, as ``packers.pack_reads`` packs them
    from pysam handles: ``paths``: kid -> indexed BAM file; ``regions``: kid -> contig -> [(start0, end0)];
    ``head_reads``: template lengths of the first N + 1 records of each file in ``table.head_tlen[kid]``.

    With ``engine`` (an ``engine.Engine``) the records are parsed on the GPU and the bulk columns decoded there: the
    table then has no ``qual`` / ``seq2`` and ``table.device_reads`` holds the ``DeviceReads`` of ``min_gt_qual``."""
    dev = engine.bam_decoder() if engine is not None else None
    parse = (lambda buf, offs, part: parse_records(buf, offs)) if dev is None else dev.parse
    kids = list(paths)
    files = {kid: (p if isinstance(p, BamFile) else BamFile(p)) for kid, p in paths.items()}
    recs = _Records(parse)
    head_tlen: Dict[str, np.ndarray] = {}
    if head_reads:
        for kid in kids:
            head_tlen[kid] = files[kid].head_tlen(head_reads + 1)
    # ---- pass 1: every merged interval of every (kid, contig), one inflate per file ----------------------------------
    plan = []                                   # (k, contig, tid or None, [(beg, end)])
    for k, kid in enumerate(kids):
        f = files[kid]
        for contig, ivs in regions.get(kid, {}).items():
            tid = f.tids.get(contig)
            iv = [(max(a, 0), max(b, 1)) for a, b in _merge(ivs)] if tid is not None else []
            plan.append((k, contig, tid, [(beg, end) for beg, end in iv if end >= beg]))
    # one read of the union of every interval's chunks per file: a chunk shared by several intervals is inflated,
    # parsed and (with an engine) copied to the device once
    kid_idx: Dict[int, np.ndarray] = {}
    for k, kid in enumerate(kids):
        qs = [(tid, beg, end) for (k2, _c, tid, iv) in plan if k2 == k for beg, end in iv]
        if qs:
            buf, offs = files[kid].fetch_union(qs)
            (kid_idx[k],) = recs.add(buf, [offs])
    allrec = lambda: np.concatenate(recs.rec) if recs.rec else np.zeros(0, dtype=L.BAM_REC_DTYPE)
    R = allrec()
    # ---- selection per (kid, contig): overlap, the duplicate rule between intervals, lone mates ----------------------
    # the packer's duplicate rule compares pysam's reference_end: bam_endpos for a mapped read with a CIGAR; for an
    # unmapped or CIGAR-less read (pysam: None) the stand-ins' pos + reference length
    ref_end = np.where(((R["flag"] & 0x4) == 0) & (R["n_cigar"] > 0), R["end"].astype(np.int64),
                       R["pos"].astype(np.int64) + R["ref_len"])
    sel_blocks = []                             # (k, contig, selected record indices before the lone mates)
    for pi, (k, contig, tid, iv) in enumerate(plan):
        parts: List[np.ndarray] = []
        if iv and k in kid_idx:
            ix_t = kid_idx[k][R["ref_id"][kid_idx[k]] == tid]            # file order = sorted by pos
            pos_t = R["pos"][ix_t].astype(np.int64)
            span = int((R["end"][ix_t].astype(np.int64) - pos_t).max()) if ix_t.shape[0] else 0
            prev_end = prev_start = None
            for beg, end in iv:
                lo = int(np.searchsorted(pos_t, beg - span, side="left"))
                hi = int(np.searchsorted(pos_t, end, side="left"))
                ix = ix_t[lo:hi]
                keep = R["end"][ix] > beg
                if prev_end is not None:
                    # a record that starts before the end of the previous (disjoint) interval came back there already
                    keep &= (R["pos"][ix] >= prev_end) | (ref_end[ix] <= prev_start)
                parts.append(ix[keep])
                prev_end, prev_start = end, beg
        sel = np.concatenate(parts) if parts else np.zeros(0, dtype=np.int64)
        sel_blocks.append([k, contig, tid, sel, None])

    def names_of(ix: np.ndarray) -> List[str]:
        nm = recs.names
        return [nm[i] for i in ix.tolist()]

    lone_req: Dict[int, list] = {}              # kid -> [(block, record index)]
    for bi, (k, contig, tid, sel, _) in enumerate(sel_blocks):
        r = R[sel]
        flag = r["flag"].astype(np.int64)
        names = names_of(sel)
        mate = _mate_join(names, flag)
        lone = np.flatnonzero((mate < 0) & ((flag & 0x1) != 0) & ((flag & 0x8) == 0) & ((flag & 0x900) == 0))
        sel_blocks[bi][4] = {(names[i], int(flag[i]) & 0xC0, int(r["pos"][i])) for i in lone.tolist()}
        # bamfile.mate() as the packer uses it: a mate on another reference is never added
        lone = lone[r["next_ref_id"][lone] == r["ref_id"][lone]]
        lone_req.setdefault(k, []).extend((bi, int(sel[i])) for i in lone.tolist())
    # ---- pass 2: one read per file of the union of the chunks at every lone mate's next_pos ---------------------------
    # Only the records chosen as mates join the load (a compact copy of their bytes): the rest of these chunks is
    # parsed once on the host and dropped, never copied to the device.
    extra: Dict[int, List[int]] = {}
    for k, reqs in lone_req.items():
        if not reqs:
            continue
        kid = kids[k]
        ri = np.array([i for _b, i in reqs], dtype=np.int64)
        rtid = R["ref_id"][ri].astype(np.int64)
        rp = np.maximum(R["next_pos"][ri].astype(np.int64), 0)
        qs = sorted(set(zip(rtid.tolist(), rp.tolist())))
        cbuf, coffs = files[kid].fetch_union([(t, p, p + 1) for t, p in qs])
        crec = parse_records(cbuf, coffs)
        # pysam's mate(): the first record in file order that overlaps the mate position and has the same name and
        # the other segment bit -- secondary and supplementary records included, as the packer gets them.  Candidates
        # are grouped by (name hash, reference) with one sort; names are compared for the few lone reads only.
        ckey = crec["name_hash"].view(np.int64)
        corder = np.lexsort((np.arange(ckey.shape[0]), crec["ref_id"], ckey))
        skey, stid = ckey[corder], crec["ref_id"][corder].astype(np.int64)
        rkey = R["name_hash"][ri].view(np.int64)
        lo = np.searchsorted(skey, rkey, side="left")
        hi = np.searchsorted(skey, rkey, side="right")
        want = np.where((R["flag"][ri] & 0x40) != 0, 0x80, 0x40)
        chosen: Dict[int, List[int]] = {}           # candidate record -> request numbers
        for q in np.flatnonzero(hi > lo).tolist():
            c = corder[lo[q]:hi[q]]
            ok = (stid[lo[q]:hi[q]] == rtid[q]) & ((crec["flag"][c] & want[q]) != 0) & \
                 (crec["pos"][c] <= rp[q]) & (crec["end"][c] > rp[q])
            c = c[ok]
            if not c.shape[0]:
                continue
            nm = recs.names[int(ri[q])]
            cn = _names(cbuf, coffs[c], crec["l_name"][c])
            m = next((int(ci) for ci, x in zip(c.tolist(), cn) if x == nm), None)
            if m is not None:
                chosen.setdefault(m, []).append(q)
        if not chosen:
            continue
        picked = np.array(sorted(chosen), dtype=np.int64)
        ln = 4 + cbuf[coffs[picked][:, None] + np.arange(4)].copy().view("<i4").reshape(-1).astype(np.int64)
        compact = gather(cbuf, coffs[picked], ln)
        (gidx,) = recs.add(compact, [np.cumsum(ln) - ln])
        R = allrec()
        global_of = dict(zip(picked.tolist(), gidx.tolist()))
        for m in picked.tolist():
            g = global_of[m]
            for q in chosen[m]:
                bi = reqs[q][0]
                blk = sel_blocks[bi]
                key = (recs.names[g], int(R["flag"][g]) & 0xC0, int(R["pos"][g]))
                extra.setdefault(bi, []).append((q, g, key))
    for bi, lst in extra.items():
        blk = sel_blocks[bi]
        keep = []
        for _q, g, key in sorted(lst):                 # in the order of the lone reads, as the packer walks them
            if key in blk[4]:
                continue
            blk[4].add(key)
            keep.append(g)
        extra[bi] = keep
    # ---- block layout: stable sort by start; reads of a block in file order among equal starts ------------------------
    contigs: List[str] = []
    cindex: Dict[str, int] = {}
    order_parts, blk_kid, blk_contig, offs_b = [], [], [], [0]
    for bi, (k, contig, tid, sel, _) in enumerate(sel_blocks):
        ix = np.concatenate([sel, np.array(extra.get(bi, []), dtype=np.int64)])
        ix = ix[np.argsort(R["pos"][ix], kind="stable")]
        if contig not in cindex:
            cindex[contig] = len(contigs)
            contigs.append(contig)
        order_parts.append(ix)
        blk_kid.append(k)
        blk_contig.append(cindex[contig])
        offs_b.append(offs_b[-1] + ix.shape[0])
    order = np.concatenate(order_parts) if order_parts else np.zeros(0, dtype=np.int64)
    recs.finish()
    r = R[order]
    n = int(order.shape[0])
    names_all = names_of(order)
    hdr = np.zeros(n, dtype=READ_HDR)
    hdr["start"], hdr["tlen"], hdr["flag"], hdr["mapq"] = r["pos"], r["tlen"], r["flag"], r["mapq"]
    hdr["aux"] = np.where(r["aux"] & 1, AUX_SAME_REF, 0) | np.where(r["aux"] & 2, AUX_HAS_SA, 0)
    ncig = r["n_cigar"].astype(np.int64)
    lens = r["l_seq"].astype(np.int64)
    hdr["n_cigar"], hdr["l_seq"] = ncig, lens
    hdr["cigar_off"] = np.cumsum(ncig) - ncig
    q0 = np.cumsum(lens) - lens
    hdr["qoff_lo"], hdr["qoff_hi"] = q0 & 0xFFFFFFFF, q0 >> 32
    src = recs.all_offs[order]
    blk_of = np.repeat(np.arange(len(offs_b) - 1, dtype=np.int32), np.diff(offs_b))
    if dev is not None:
        # mates on the device (unfz_bam_mate_join); the reads it leaves to the host are resolved by name in their block
        dev.prepare(src)
        mate = resolve_left_mates(dev.mate_join(r["name_hash"], blk_of, r["flag"].astype(np.int32)), names_all,
                                  r["flag"], np.asarray(offs_b))
    else:
        mate = np.full(n, -1, dtype=np.int64)
        for b in range(len(offs_b) - 1):
            lo, hi = offs_b[b], offs_b[b + 1]
            m = _mate_join(names_all[lo:hi], hdr["flag"][lo:hi].astype(np.int64))
            mate[lo:hi] = np.where(m >= 0, m + lo, -1)
    hdr["mate"] = mate
    # ---- bulk columns --------------------------------------------------------------------------------------------------
    lname = r["l_name"].astype(np.int64)
    cig_src = src + 36 + lname
    cigar = recs.gather(cig_src, 4 * ncig).view("<u4")
    table = ReadTable(kids=kids, contigs=contigs, blk_kid=np.array(blk_kid, dtype=np.int32),
                      blk_contig=np.array(blk_contig, dtype=np.int32), blk_off=np.array(offs_b, dtype=np.int64),
                      hdr=hdr, cigar=cigar, qual=None, seq2=None, names=names_all)
    table.head_tlen = head_tlen
    if dev is not None:
        table.n_bases = int(lens.sum())
        table.device_source = dev
        table.device_reads = dev.emit(table, min_gt_qual)
        table.validate()
        return table
    buf = recs.buffer()
    seq_src = cig_src + 4 * ncig
    sb = (lens + 1) // 2
    packed = gather(buf, seq_src, sb)
    nib = np.empty(2 * packed.shape[0], dtype=np.uint8)
    nib[0::2], nib[1::2] = packed >> 4, packed & 15
    odd = np.flatnonzero(lens & 1)
    if odd.shape[0]:
        pad = (np.cumsum(2 * sb) - 1)[odd]               # the unused low nibble of the last byte of an odd-length read
        nib = np.delete(nib, pad)
    qb = gather(buf, seq_src + sb, lens)
    missing = np.zeros(n, dtype=bool)
    nz = lens > 0
    missing[nz] = buf[(seq_src + sb)[nz]] == 0xFF
    if missing.any():
        qb[np.repeat(missing, lens)] = 0
    esc = _NIB_ESC[nib]
    table.qual = np.where(esc, qb | QUAL_ESCAPE, qb & 0x7F).astype(np.uint8)
    table.seq2 = pack_seq(_NIB_CODE[nib])
    table.validate()
    return table


# ------------------------------------------------------------------------------------------------
# writer
# ------------------------------------------------------------------------------------------------

def encode_tag(tag: str, typ: str, value) -> bytes:
    """One aux field in BAM encoding (types A c C s S i I f Z H B; B takes (subtype, values))."""
    t = tag.encode() + typ.encode()
    if typ == "A":
        return t + value.encode()
    if typ in "cCsSiIf":
        return t + struct.pack("<" + {"c": "b", "C": "B", "s": "h", "S": "H", "i": "i", "I": "I", "f": "f"}[typ], value)
    if typ in "ZH":
        return t + value.encode() + b"\0"
    if typ == "B":
        sub, vals = value
        fmt = {"c": "b", "C": "B", "s": "h", "S": "H", "i": "i", "I": "I", "f": "f"}[sub]
        return t + sub.encode() + struct.pack("<I", len(vals)) + struct.pack("<%d%s" % (len(vals), fmt), *vals)
    raise ValueError("unknown aux type %r" % typ)


def write_bam(table: ReadTable, kid: int, path: str, extra_tags: Optional[Dict[int, bytes]] = None,
              missing_qual: Optional[np.ndarray] = None, other_ref: Optional[np.ndarray] = None,
              ref_lens: Optional[Dict[str, int]] = None, level: int = 6, chunk_reads: int = 1 << 18,
              common_tags: bytes = b"", index: str = "bai") -> None:
    """Coordinate-sorted BAM + index of kid ``kid``'s reads of ``table``: ``path + ".bai"``, or with ``index="csi"``
    ``path + ".csi"`` (min_shift 14, depth 5, as ``samtools index -c`` writes it).

    References: ``table.contigs`` in table order (a contig without reads of this kid is an empty reference).  Names:
    ``table.names`` or the synthesized pair names.  Bases: A C G T as they are; an escaped code 0 is N and an escaped
    code 1 one of ``=MRSVWYHKDB`` (cycling with the base index).  The mate position is the mate row's start; a paired
    read without a mate row gets its own start, so a mate lookup finds nothing.  next_refID is refID when the read has
    AUX_SAME_REF, else -1 (or the next reference for reads in ``other_ref``).  Reads with AUX_HAS_SA get an SA tag.
    ``extra_tags``: read index -> encoded aux bytes appended (``encode_tag``); ``missing_qual``: read indices written
    with a missing quality string (0xFF); ``common_tags``: encoded aux bytes appended to every record."""
    t = table
    blocks = [b for b in range(t.n_blocks) if int(t.blk_kid[b]) == kid]
    blocks.sort(key=lambda b: int(t.blk_contig[b]))
    rows = np.concatenate([np.arange(t.blk_off[b], t.blk_off[b + 1]) for b in blocks]) if blocks else np.zeros(0, np.int64)
    tid_of_row = np.concatenate([np.full(int(t.blk_off[b + 1] - t.blk_off[b]), int(t.blk_contig[b]), np.int32)
                                 for b in blocks]) if blocks else np.zeros(0, np.int32)
    ends = t.ref_ends()
    n_ref = len(t.contigs)
    lens_ref = []
    for c, name in enumerate(t.contigs):
        m = ends[rows[tid_of_row == c]] if rows.shape[0] else np.zeros(0)
        lens_ref.append(int((ref_lens or {}).get(name, max(int(m.max()) + 1000 if m.shape[0] else 1000, 1))))
    text = b"@HD\tVN:1.6\tSO:coordinate\n" + b"".join(b"@SQ\tSN:%s\tLN:%d\n" % (nm.encode(), ln)
                                                      for nm, ln in zip(t.contigs, lens_ref))
    head = bytearray(b"BAM\x01" + struct.pack("<i", len(text)) + text + struct.pack("<i", n_ref))
    for nm, ln in zip(t.contigs, lens_ref):
        head += struct.pack("<i", len(nm) + 1) + nm.encode() + b"\0" + struct.pack("<i", ln)
    missing = np.zeros(t.n_reads, dtype=bool)
    if missing_qual is not None:
        missing[np.asarray(missing_qual, dtype=np.int64)] = True
    other = np.zeros(t.n_reads, dtype=bool)
    if other_ref is not None:
        other[np.asarray(other_ref, dtype=np.int64)] = True
    extra_tags = extra_tags or {}
    nib_of_code = np.array([1, 2, 4, 8], dtype=np.uint8)
    iupac = np.frombuffer(bytes([_NIB_CHARS.index(ch) for ch in b"=MRSVWYHKDB"]), dtype=np.uint8)
    out_blocks: List[bytes] = []
    # records: serialised in chunks of reads; every record's start is remembered as an uncompressed stream offset
    rec_start = np.zeros(rows.shape[0] + 1, dtype=np.int64)
    stream: List[bytes] = []
    pos_u = 0
    for a in range(0, rows.shape[0], chunk_reads):
        rr = rows[a: a + chunk_reads]
        h = t.hdr[rr]
        m = rr.shape[0]
        tid = tid_of_row[a: a + m]
        names = [nm.encode() for nm in t.names_of(rr)]
        lname = np.fromiter((len(x) + 1 for x in names), dtype=np.int64, count=m)
        ncig = h["n_cigar"].astype(np.int64)
        L_ = h["l_seq"].astype(np.int64)
        q0 = h["qoff_lo"].astype(np.int64) | (h["qoff_hi"].astype(np.int64) << 32)
        # aux: SA for reads with the bit, then the caller's tags
        aux = []
        for j, r_ in enumerate(rr.tolist()):
            x = b""
            if int(h["aux"][j]) & AUX_HAS_SA:
                x += encode_tag("SA", "Z", "%s,%d,+,%dM,60,0;" % (t.contigs[int(tid[j])], int(h["start"][j]) + 1, max(int(L_[j]), 1)))
            x += extra_tags.get(r_, b"") + common_tags
            aux.append(x)
        laux = np.fromiter(map(len, aux), dtype=np.int64, count=m)
        sb = (L_ + 1) // 2
        size = 36 + lname + 4 * ncig + sb + L_ + laux
        fx = np.zeros(m, dtype=_FIXED)
        fx["block_size"] = size - 4
        fx["ref_id"] = tid
        fx["pos"] = h["start"]
        fx["l_name"] = lname
        fx["mapq"] = h["mapq"]
        fx["n_cigar"] = ncig
        fx["flag"] = h["flag"]
        fx["l_seq"] = L_
        fx["tlen"] = h["tlen"]
        e = ends[rr]
        fx["bin"] = [reg2bin(int(s), int(max(en, s + 1))) for s, en in zip(h["start"].tolist(), e.tolist())]
        mrow = h["mate"].astype(np.int64)
        same = (h["aux"] & AUX_SAME_REF) != 0
        fx["next_ref_id"] = np.where(same, tid, np.where(other[rr], (tid + 1) % max(n_ref, 1), -1))
        fx["next_pos"] = np.where(mrow >= 0, t.hdr["start"][np.maximum(mrow, 0)], h["start"])
        # bases and qualities of the chunk
        gidx = _ranges(q0, L_)
        code = (t.seq2[gidx >> 2] >> ((gidx & 3) << 1).astype(np.uint8)) & 3
        qual = t.qual[gidx]
        escm = (qual & QUAL_ESCAPE) != 0
        nib = np.where(escm, np.where(code == 0, 15, iupac[gidx % iupac.shape[0]]), nib_of_code[code]).astype(np.uint8)
        qv = (qual & 0x7F).astype(np.uint8)
        rep_missing = np.repeat(missing[rr], L_)
        qv[rep_missing] = 0xFF
        # pad odd reads with a zero nibble, then pack two per byte
        padded = np.zeros(int((2 * sb).sum()), dtype=np.uint8)
        pstart = np.cumsum(2 * sb) - 2 * sb
        padded[np.repeat(pstart - (np.cumsum(L_) - L_), L_) + np.arange(int(L_.sum()))] = nib
        seqb = (padded[0::2] << 4) | padded[1::2]
        cig = t.cigar[_ranges(h["cigar_off"].astype(np.int64), ncig)]
        # one source blob, then every record as six ranges of it
        blobs = [fx.view(np.uint8), np.frombuffer(b"\0".join(names) + b"\0", dtype=np.uint8),
                 cig.astype("<u4").view(np.uint8), seqb, qv, np.frombuffer(b"".join(aux), dtype=np.uint8)]
        base = np.cumsum([0] + [bb.shape[0] for bb in blobs])
        src_blob = np.concatenate(blobs)
        seg_len = np.stack([np.full(m, 36), lname, 4 * ncig, sb, L_, laux], axis=1)
        seg_src = np.stack([base[i] + np.cumsum(seg_len[:, i]) - seg_len[:, i] for i in range(6)], axis=1)
        data = gather(src_blob, seg_src.reshape(-1), seg_len.reshape(-1))
        rec_start[a + 1: a + m + 1] = pos_u + np.cumsum(size)
        pos_u += int(size.sum())
        stream.append(data.tobytes())
    voff = write_bgzf(path, bytes(head), b"".join(stream), level)
    cols = (n_ref, tid_of_row, t.hdr["start"][rows].astype(np.int64), ends[rows], voff(rec_start[:-1]),
            voff(rec_start[1:]))
    if index == "csi":
        write_csi(path + ".csi", *cols)
    elif index == "bai":
        _write_bai(path + ".bai", *cols)
    else:
        raise ValueError("index must be 'bai' or 'csi', not %r" % index)


def write_bgzf(path: str, head: bytes, body: bytes, level: int = 6):
    """``head`` and ``body`` BGZF-compressed into ``path`` (the header in blocks of its own, as htslib writes it), plus the
    EOF block.  Returns the map of uncompressed body offsets (an array) to virtual file offsets."""
    head_blocks = [head[i: i + _BLOCK_IN] for i in range(0, len(head), _BLOCK_IN)] or [b""]
    body_blocks = [body[i: i + _BLOCK_IN] for i in range(0, len(body), _BLOCK_IN)]
    with ThreadPoolExecutor(_THREADS) as pool:
        comp = list(pool.map(lambda raw: _bgzf_block(raw, level), head_blocks + body_blocks))
    coff = np.cumsum([0] + [len(c) for c in comp])
    body_coff = coff[len(head_blocks):]                     # file offset of each body block (and of the EOF block)
    with open(path, "wb") as f:
        for c in comp:
            f.write(c)
        f.write(BGZF_EOF)

    def voff(u: np.ndarray) -> np.ndarray:
        blk = u // _BLOCK_IN
        return (body_coff[blk].astype(np.uint64) << np.uint64(16)) | (u % _BLOCK_IN).astype(np.uint64)
    return voff


def _ranges(start: np.ndarray, length: np.ndarray) -> np.ndarray:
    """Concatenation of arange(start[i], start[i] + length[i])."""
    tot = int(length.sum())
    return np.repeat(start - (np.cumsum(length) - length), length) + np.arange(tot, dtype=np.int64)


def _write_bai(path: str, n_ref: int, tid: np.ndarray, pos: np.ndarray, end_raw: np.ndarray, vbeg: np.ndarray,
               vend: np.ndarray) -> None:
    """BAI of records sorted by (tid, pos)."""
    with open(path, "wb") as f:
        f.write(b"BAI\x01" + struct.pack("<i", n_ref) + index_refs(n_ref, tid, pos, end_raw, vbeg, vend))


def index_refs(n_ref: int, tid: np.ndarray, pos: np.ndarray, end_raw: np.ndarray, vbeg: np.ndarray,
               vend: np.ndarray) -> bytes:
    """The per-reference part of a BAI or TBI for records sorted by (tid, pos) spanning [pos, end_raw) at virtual offsets
    [vbeg, vend): per reference the bins (chunks of consecutive records of the same bin merged), the pseudo-bin of counts
    and the 16 kb linear index; then the count of records without a coordinate (0)."""
    end = np.maximum(end_raw, pos + 1)
    out = bytearray()
    for t in range(n_ref):
        sel = np.flatnonzero(tid == t)
        bins: Dict[int, List[List[int]]] = {}
        lin: Dict[int, int] = {}
        for i in sel.tolist():
            b = reg2bin(int(pos[i]), int(end[i]))
            ch = bins.setdefault(b, [])
            vb, ve = int(vbeg[i]), int(vend[i])
            if ch and ch[-1][1] == vb:
                ch[-1][1] = ve
            else:
                ch.append([vb, ve])
            for w in range(int(pos[i]) >> 14, ((int(end[i]) - 1) >> 14) + 1):
                if w not in lin:
                    lin[w] = vb
        nb = len(bins) + (1 if sel.shape[0] else 0)
        out += struct.pack("<i", nb)
        for b in sorted(bins):
            out += struct.pack("<Ii", b, len(bins[b]))
            for vb, ve in bins[b]:
                out += struct.pack("<QQ", vb, ve)
        if sel.shape[0]:
            out += struct.pack("<Ii", 37450, 2) + struct.pack("<QQ", int(vbeg[sel[0]]), int(vend[sel[-1]]))
            out += struct.pack("<QQ", sel.shape[0], 0)
        n_intv = (max(lin) + 1) if lin else 0
        vals, last = [], 0
        for w in range(n_intv):
            last = lin.get(w, last)
            vals.append(last)
        out += struct.pack("<i", n_intv) + struct.pack("<%dQ" % n_intv, *vals)
    out += struct.pack("<Q", 0)
    return bytes(out)


def csi_depth(max_end: int, min_shift: int = 14) -> int:
    """The smallest depth (at least 5) whose binning spans [0, max_end), as htslib sizes a CSI."""
    depth = 5
    while (1 << (min_shift + 3 * depth)) < max_end:
        depth += 1
    return depth


def write_csi(path: str, n_ref: int, tid: np.ndarray, pos: np.ndarray, end_raw: np.ndarray, vbeg: np.ndarray,
              vend: np.ndarray, min_shift: int = 14, depth: Optional[int] = None, aux: bytes = b"",
              level: int = 6) -> None:
    """CSI (BGZF-compressed) of records sorted by (tid, pos) spanning [pos, end_raw) at virtual offsets [vbeg, vend).
    ``depth`` None: the smallest that spans the records.  ``aux``: the tabix header of a .vcf.gz index, empty for BCF and
    BAM."""
    if depth is None:
        depth = csi_depth(int(np.max(np.maximum(end_raw, pos + 1))) if len(pos) else 1, min_shift)
    body = (b"CSI\x01" + struct.pack("<3i", min_shift, depth, len(aux)) + aux + struct.pack("<i", n_ref)
            + csi_refs(n_ref, tid, pos, end_raw, vbeg, vend, min_shift, depth))
    write_bgzf(path, body, b"", level)


def csi_refs(n_ref: int, tid: np.ndarray, pos: np.ndarray, end_raw: np.ndarray, vbeg: np.ndarray, vend: np.ndarray,
             min_shift: int, depth: int) -> bytes:
    """The per-reference part of a CSI: per reference the bins (chunks of consecutive records of the same bin merged)
    with their ``loffset`` -- the virtual offset of the first record that ends after the bin's start, so no record before
    it overlaps the bin -- and the pseudo-bin of counts; then the count of records without a coordinate (0)."""
    tid = np.asarray(tid, dtype=np.int64)
    pos = np.asarray(pos, dtype=np.int64)
    end = np.maximum(np.asarray(end_raw, dtype=np.int64), pos + 1)
    out = bytearray()
    for t in range(n_ref):
        sel = np.flatnonzero(tid == t)
        bins: Dict[int, List[List[int]]] = {}
        for i in sel.tolist():
            b = reg2bin(int(pos[i]), int(end[i]), min_shift, depth)
            ch = bins.setdefault(b, [])
            vb, ve = int(vbeg[i]), int(vend[i])
            if ch and ch[-1][1] == vb:
                ch[-1][1] = ve
            else:
                ch.append([vb, ve])
        run_end = np.maximum.accumulate(end[sel]) if sel.shape[0] else end[sel]
        out += struct.pack("<i", len(bins) + (1 if sel.shape[0] else 0))
        for b in sorted(bins):
            lvl = next(l for l in range(depth, -1, -1) if b >= bin_first(l))
            start = (b - bin_first(lvl)) << (min_shift + 3 * (depth - lvl))
            first = int(np.searchsorted(run_end, start, side="right"))
            loff = int(vbeg[sel[first]]) if first < sel.shape[0] else 0
            out += struct.pack("<IQi", b, loff, len(bins[b]))
            for vb, ve in bins[b]:
                out += struct.pack("<QQ", vb, ve)
        if sel.shape[0]:
            out += struct.pack("<IQi", pseudo_bin(depth), 0, 2) + struct.pack("<QQ", int(vbeg[sel[0]]), int(vend[sel[-1]]))
            out += struct.pack("<QQ", sel.shape[0], 0)
    out += struct.pack("<Q", 0)
    return bytes(out)
