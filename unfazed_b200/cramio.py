"""Indexed CRAM 3.0 files without pysam: CRAI queries and block decompression on the host, slice decoding to BAM records
in native code.

* ``CramFile`` -- one CRAM 3.0 file, its ``.crai`` and a plain FASTA reference (``.fai``, or an index built in memory by
  one scan).  It answers the calls ``bamio.read_regions`` makes on a ``BamFile``: ``tids``, ``refs``,
  ``fetch_union(queries) -> (buf, offs)`` and ``head_tlen(n)``.  ``buf`` holds BAM records (block_size ... aux), so
  everything downstream of the decode -- overlap selection, duplicates between intervals, lone mates, the device parse,
  the mate join and the planes -- is the BAM path.  CRAI entries select the slices; containers and slice headers are
  parsed here, every container header and block checked against its CRC32, and the blocks of the selected slices are
  decompressed in a thread pool (raw, gzip, bzip2, lzma through the standard library, rANS 4x8 natively).  Each slice
  is flattened into an ``UnfzCramSlice`` descriptor; csrc/cram.cu decodes it (host entry points, or the GPU with an
  engine).
* ``write_cram`` -- a sorted CRAM 3.0 + ``.crai`` from a ``ReadTable`` (tests and tools), with the block method, the
  encodings, slice sizes, multi-reference slices, an embedded reference and RR = false chosen by options.
* ``rans_encode`` -- rANS 4x8 order 0 / 1 (the writer's method 4, and the tests' encoder).

Malformed input raises ``ValueError`` naming the file and the byte offset of the container.
"""
from __future__ import annotations

import bz2
import ctypes as C
import gzip
import hashlib
import heapq
import lzma
import mmap
import os
import struct
import tempfile
import zlib
from concurrent.futures import ThreadPoolExecutor
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import _lib as L
from . import bamio

SERIES = ["BF", "CF", "RI", "RL", "AP", "RG", "RN", "MF", "NS", "NP", "TS", "NF", "TL", "FN", "FC", "FP", "DL", "BB",
          "QQ", "BS", "IN", "RS", "PD", "HC", "SC", "MQ", "BA", "QS"]
_ARRAY_SERIES = {"RN", "BB", "QQ", "IN", "SC"}
E_NULL, E_EXTERNAL, E_GOLOMB, E_HUFFMAN, E_BYTE_ARRAY_LEN, E_BYTE_ARRAY_STOP, E_BETA, E_SUBEXP, E_GOLOMB_RICE, E_GAMMA = range(10)
METHODS = {"raw": 0, "gzip": 1, "bzip2": 2, "lzma": 3, "rans0": 4, "rans1": 4}
EOF_START = 4542278                       # the EOF container's alignment start ("EOF" in ITF8 bytes)
_THREADS = min(32, os.cpu_count() or 4)

SLICE_DTYPE = np.dtype([("core_off", "<i8"), ("core_len", "<i8"), ("ext_off", "<i8"), ("prog_off", "<i8"),
                        ("refs_off", "<i8"), ("rec_first", "<i8"), ("rg_off", "<i8"), ("n_ext", "<i4"),
                        ("n_records", "<i4"), ("n_refs", "<i4"), ("ref_id", "<i4"), ("ap_start", "<i4"), ("flags", "<i4"),
                        ("sub", "u1", (5,)), ("_pad", "u1", (3,))])
EXT_DTYPE = np.dtype([("off", "<i8"), ("len", "<i8")])
REF_DTYPE = np.dtype([("off", "<i8"), ("start", "<i8"), ("len", "<i8"), ("ref_id", "<i4"), ("_pad", "<i4")])
assert SLICE_DTYPE.itemsize == 88 and EXT_DTYPE.itemsize == 16 and REF_DTYPE.itemsize == 32
AP_DELTA = 0x1
STATUS = {1: "a stream overruns its block", 2: "a data series has no usable encoding or block", 3: "a value is out of range"}


def _ptr(a: np.ndarray) -> int:
    return a.ctypes.data


# ------------------------------------------------------------------------------------------------
# ITF8 / LTF8
# ------------------------------------------------------------------------------------------------

def itf8(v: int) -> bytes:
    v &= 0xFFFFFFFF
    if v < 0x80:
        return bytes([v])
    if v < 0x4000:
        return bytes([0x80 | (v >> 8), v & 0xFF])
    if v < 0x200000:
        return bytes([0xC0 | (v >> 16), (v >> 8) & 0xFF, v & 0xFF])
    if v < 0x10000000:
        return bytes([0xE0 | (v >> 24), (v >> 16) & 0xFF, (v >> 8) & 0xFF, v & 0xFF])
    return bytes([0xF0 | (v >> 28), (v >> 20) & 0xFF, (v >> 12) & 0xFF, (v >> 4) & 0xFF, v & 0x0F])


def ltf8(v: int) -> bytes:
    v &= 0xFFFFFFFFFFFFFFFF
    for n in range(1, 9):                    # n bytes: n - 1 leading one bits, 7 * n payload bits
        if v < (1 << (7 * n)) and n < 8:
            lead = (0xFF << (8 - (n - 1))) & 0xFF
            return bytes([lead | (v >> (8 * (n - 1)))]) + v.to_bytes(8, "big")[8 - (n - 1):]
    if v < (1 << 56):
        return b"\xFE" + v.to_bytes(7, "big")
    return b"\xFF" + v.to_bytes(8, "big")


class _Reader:
    """ITF8 / LTF8 / fixed-width reads over bytes; raises _Short past the end."""

    def __init__(self, d, p: int = 0, end: Optional[int] = None):
        self.d, self.p = d, p
        self.end = len(d) if end is None else end

    def byte(self) -> int:
        if self.p >= self.end:
            raise _Short()
        b = self.d[self.p]
        self.p += 1
        return b

    def take(self, n: int) -> bytes:
        if n < 0 or self.p + n > self.end:
            raise _Short()
        b = bytes(self.d[self.p:self.p + n])
        self.p += n
        return b

    def i32(self) -> int:
        return struct.unpack("<i", self.take(4))[0]

    def itf8(self) -> int:
        b0 = self.byte()
        if b0 < 0x80:
            v = b0
        elif b0 < 0xC0:
            v = ((b0 & 0x3F) << 8) | self.byte()
        elif b0 < 0xE0:
            v = ((b0 & 0x1F) << 16) | (self.byte() << 8) | self.byte()
        elif b0 < 0xF0:
            v = ((b0 & 0x0F) << 24) | (self.byte() << 16) | (self.byte() << 8) | self.byte()
        else:
            v = ((b0 & 0x0F) << 28) | (self.byte() << 20) | (self.byte() << 12) | (self.byte() << 4) | (self.byte() & 0x0F)
        return v - (1 << 32) if v >= (1 << 31) else v

    def ltf8(self) -> int:
        b0 = self.byte()
        n = 0
        while n < 8 and b0 & (0x80 >> n):
            n += 1
        if n == 8:
            return int.from_bytes(self.take(8), "big")
        v = b0 & (0xFF >> (n + 1)) if n < 7 else 0
        for _ in range(n):
            v = (v << 8) | self.byte()
        return v

    def itf8_array(self) -> List[int]:
        return [self.itf8() for _ in range(self.itf8())]


class _Short(Exception):
    pass


# ------------------------------------------------------------------------------------------------
# rANS 4x8
# ------------------------------------------------------------------------------------------------

def _normalise(counts: np.ndarray) -> np.ndarray:
    """Frequencies summing to 4096 with every present symbol at least 1."""
    tot = int(counts.sum())
    f = np.zeros(256, dtype=np.int64)
    nz = np.flatnonzero(counts)
    f[nz] = np.maximum(1, counts[nz] * 4096 // tot)
    f[nz[np.argmax(f[nz])]] += 4096 - int(f.sum())
    if f.min() < 0 or int(f[nz].min()) < 1:                 # the largest could not absorb the rounding: flatten
        f[nz] = 1
        f[nz[0]] += 4096 - len(nz)
    return f


def _freq_table(f: np.ndarray) -> bytes:
    out = bytearray()
    rle = 0
    for j in range(256):
        if not f[j]:
            continue
        if rle:
            rle -= 1
        else:
            out.append(j)
            if j and f[j - 1]:
                r = j + 1
                while r < 256 and f[r]:
                    r += 1
                rle = r - (j + 1)
                out.append(rle)
        v = int(f[j])
        out += bytes([v]) if v < 128 else bytes([0x80 | (v >> 8), v & 0xFF])
    out.append(0)
    return bytes(out)


def rans_encode(data: bytes, order: int = 0) -> bytes:
    """rANS 4x8 of ``data`` (CRAM block method 4), order 0 or 1, as htslib's rANS_static lays it out."""
    data = bytes(data)
    n = len(data)
    if n == 0:
        return bytes([order]) + struct.pack("<II", 0, 0)
    a = np.frombuffer(data, dtype=np.uint8)
    Lr = 1 << 23
    if order == 0:
        F = _normalise(np.bincount(a, minlength=256))
        Cc = np.concatenate([[0], np.cumsum(F)[:-1]])
        table = _freq_table(F)
        steps = [(i & 3, data[i], 0) for i in range(n)]            # (lane, symbol, context)
        Fx, Cx = {0: F}, {0: Cc}
    else:
        q = n >> 2
        ctx = np.zeros(n, dtype=np.int64)
        lanes = [list(range(k * q, (k + 1) * q)) for k in range(4)]
        lanes[3] += list(range(4 * q, n))
        for lane in lanes:
            prev = 0
            for i in lane:
                ctx[i] = prev
                prev = data[i]
        Fx, Cx = {}, {}
        table = bytearray()
        used = sorted(set(ctx.tolist()))
        rle = 0
        for i in used:
            F = _normalise(np.bincount(a[ctx == i], minlength=256))
            Fx[i], Cx[i] = F, np.concatenate([[0], np.cumsum(F)[:-1]])
        present = np.zeros(256, dtype=bool)
        present[used] = True
        for i in range(256):
            if not present[i]:
                continue
            if rle:
                rle -= 1
            else:
                table.append(i)
                if i and present[i - 1]:
                    r = i + 1
                    while r < 256 and present[r]:
                        r += 1
                    rle = r - (i + 1)
                    table.append(rle)
            table += _freq_table(Fx[i])
        table.append(0)
        table = bytes(table)
        order_ix = []
        for j in range(q):
            for k in range(4):
                order_ix.append(j + k * q)
        order_ix += list(range(4 * q, n))
        steps = [(3 if (q == 0 or i >= 4 * q) else i // q, data[i], int(ctx[i])) for i in order_ix]
    R = [Lr] * 4
    out = bytearray()                       # emitted bytes, reversed at the end
    for lane, s, c in reversed(steps):
        f, st = int(Fx[c][s]), int(Cx[c][s])
        x = R[lane]
        x_max = ((Lr >> 12) << 8) * f
        while x >= x_max:
            out.append(x & 0xFF)
            x >>= 8
        R[lane] = ((x // f) << 12) + (x % f) + st
    body = struct.pack("<4I", *R) + bytes(reversed(out))
    payload = table + body
    return bytes([order]) + struct.pack("<II", len(payload), n) + payload


def rans_decode(data: bytes) -> bytes:
    """rANS 4x8 decode (native)."""
    src = np.frombuffer(bytes(data), dtype=np.uint8)
    if src.shape[0] < 9:
        raise ValueError("rANS stream shorter than its header")
    raw = struct.unpack_from("<I", bytes(data), 5)[0]
    out = np.empty(max(raw, 1), dtype=np.uint8)
    got = L.load().unfz_rans4x8_decode_host(_ptr(src), int(src.shape[0]), _ptr(out), int(raw))
    if got != raw:
        raise ValueError("malformed rANS 4x8 stream")
    return out[:raw].tobytes()


def _compress(raw: bytes, method: str) -> Tuple[int, bytes]:
    if method == "raw":
        return 0, raw
    if method == "gzip":
        return 1, gzip.compress(raw, 6, mtime=0)
    if method == "bzip2":
        return 2, bz2.compress(raw)
    if method == "lzma":
        return 3, lzma.compress(raw)
    if method in ("rans0", "rans1"):
        return 4, rans_encode(raw, 0 if method == "rans0" else 1)
    raise ValueError("unknown block method %r" % method)


def _decompress(method: int, data: bytes, raw_size: int) -> bytes:
    if method == 0:
        out = data
    elif method == 1:
        out = gzip.decompress(data)
    elif method == 2:
        out = bz2.decompress(data)
    elif method == 3:
        out = lzma.decompress(data)
    elif method == 4:
        out = rans_decode(data)
    else:
        raise ValueError("unknown block compression method %d" % method)
    if len(out) != raw_size:
        raise ValueError("block decompresses to %d bytes, its header says %d" % (len(out), raw_size))
    return out


# ------------------------------------------------------------------------------------------------
# containers and blocks
# ------------------------------------------------------------------------------------------------

def block_bytes(method: int, ctype: int, cid: int, raw_size: int, data: bytes) -> bytes:
    b = bytes([method, ctype]) + itf8(cid) + itf8(len(data)) + itf8(raw_size) + data
    return b + struct.pack("<I", zlib.crc32(b))


def container_bytes(ref_id: int, start: int, span: int, n_rec: int, counter: int, bases: int, n_blocks: int,
                    landmarks: Sequence[int], body: bytes) -> bytes:
    h = (struct.pack("<i", len(body)) + itf8(ref_id) + itf8(start) + itf8(span) + itf8(n_rec) + ltf8(counter)
         + ltf8(bases) + itf8(n_blocks) + itf8(len(landmarks)) + b"".join(itf8(x) for x in landmarks))
    return h + struct.pack("<I", zlib.crc32(h)) + body


EOF_CONTAINER = container_bytes(-1, EOF_START, 0, 0, 0, 0, 1, [], block_bytes(0, 1, 0, 6, b"\x01\x00\x01\x00\x01\x00"))


class _Block:
    __slots__ = ("method", "ctype", "cid", "size", "raw_size", "data_off", "end")


class _Container:
    __slots__ = ("off", "ref_id", "start", "span", "n_rec", "counter", "n_blocks", "landmarks", "data_off", "length",
                 "comp")


# ------------------------------------------------------------------------------------------------
# reference
# ------------------------------------------------------------------------------------------------

class Fasta:
    """A plain-text FASTA through its ``.fai`` (or an index built by one scan, kept in memory)."""

    def __init__(self, path: str):
        self.path = path
        with open(path, "rb") as f:
            size = os.fstat(f.fileno()).st_size
            self.data = mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ) if size else b""
        if self.data[:2] == b"\x1f\x8b":
            raise ValueError("%s: a compressed FASTA is not read natively" % path)
        self.index: Dict[str, Tuple[int, int, int, int]] = {}
        fai = path + ".fai"
        if os.path.exists(fai):
            for line in open(fai):
                f = line.rstrip("\n").split("\t")
                if len(f) >= 5:
                    self.index[f[0]] = (int(f[1]), int(f[2]), int(f[3]), int(f[4]))
        else:
            self._scan()

    def _scan(self):
        d, p, n = self.data, 0, len(self.data)
        while p < n:
            if d[p:p + 1] != b">":
                raise ValueError("%s: not a FASTA file (byte %d)" % (self.path, p))
            e = d.find(b"\n", p)
            e = n if e < 0 else e
            name = bytes(d[p + 1:e]).split()[0].decode()
            off = e + 1
            length, linebases, linewidth, q = 0, 0, 0, off
            while q < n and d[q:q + 1] != b">":
                le = d.find(b"\n", q)
                le = n if le < 0 else le
                line = bytes(d[q:le]).rstrip(b"\r")
                if not linebases:
                    linebases, linewidth = len(line), le + 1 - q
                length += len(line)
                q = le + 1
            self.index[name] = (length, off, linebases, linewidth)
            p = q

    def length(self, name: str) -> int:
        return self.index[name][0]

    def fetch(self, name: str, beg: int, end: int) -> bytes:
        """Bases [beg, end) (0-based) of ``name``, upper case, clipped to the sequence."""
        ln, off, lb, lw = self.index[name]
        beg, end = max(beg, 0), min(end, ln)
        if end <= beg:
            return b""
        a = off + (beg // lb) * lw + beg % lb
        b = off + ((end - 1) // lb) * lw + (end - 1) % lb + 1
        return bytes(self.data[a:b]).replace(b"\n", b"").replace(b"\r", b"").upper()


def is_plain_fasta(path: Optional[str]) -> bool:
    if not path or not os.path.isfile(path):
        return False
    with open(path, "rb") as f:
        return f.read(1) == b">"


# ------------------------------------------------------------------------------------------------
# reader
# ------------------------------------------------------------------------------------------------

def index_path(path: str) -> Optional[str]:
    """``<file>.crai``, or ``<stem>.crai`` when that is missing."""
    for p in (path + ".crai", os.path.splitext(path)[0] + ".crai"):
        if os.path.exists(p):
            return p
    return None


def file_version(path: str) -> Optional[Tuple[int, int]]:
    """(major, minor) of the file definition, or None for a file that is not CRAM."""
    with open(path, "rb") as f:
        head = f.read(6)
    return (head[4], head[5]) if len(head) == 6 and head[:4] == b"CRAM" else None


def _parse_encoding(r: _Reader) -> tuple:
    codec = r.itf8()
    size = r.itf8()
    p = _Reader(r.take(size))
    if codec == E_NULL:
        return (E_NULL,)
    if codec == E_EXTERNAL:
        return (E_EXTERNAL, p.itf8())
    if codec == E_HUFFMAN:
        return (E_HUFFMAN, p.itf8_array(), p.itf8_array())
    if codec == E_BYTE_ARRAY_LEN:
        return (E_BYTE_ARRAY_LEN, _parse_encoding(p), _parse_encoding(p))
    if codec == E_BYTE_ARRAY_STOP:
        return (E_BYTE_ARRAY_STOP, p.byte(), p.itf8())
    if codec in (E_BETA, E_SUBEXP):
        return (codec, p.itf8(), p.itf8())
    if codec == E_GAMMA:
        return (E_GAMMA, p.itf8())
    if codec in (E_GOLOMB, E_GOLOMB_RICE):
        raise ValueError("GOLOMB%s encoding is not supported" % ("_RICE" if codec == E_GOLOMB_RICE else ""))
    raise ValueError("unknown encoding %d" % codec)


class _CompHeader:
    """The compression header of one container: preservation map, data series encodings, tag dictionary and encodings."""

    def __init__(self, data: bytes):
        r = _Reader(data)
        self.rn, self.ap_delta, self.rr = True, True, True
        self.sub = bytes([0x1B] * 5)
        self.td: List[List[int]] = [[]]
        size = r.itf8()
        p = _Reader(r.take(size))
        for _ in range(p.itf8()):
            k = p.take(2)
            if k == b"RN":
                self.rn = bool(p.byte())
            elif k == b"AP":
                self.ap_delta = bool(p.byte())
            elif k == b"RR":
                self.rr = bool(p.byte())
            elif k == b"SM":
                self.sub = p.take(5)
            elif k == b"TD":
                raw = p.take(p.itf8())
                lines = raw.split(b"\0")
                if lines and lines[-1] == b"":
                    lines = lines[:-1]
                self.td = [[(ln[i] << 16) | (ln[i + 1] << 8) | ln[i + 2] for i in range(0, len(ln) - 2, 3)] for ln in lines]
            else:
                raise ValueError("unknown preservation map key %r" % k)
        size = r.itf8()
        p = _Reader(r.take(size))
        self.series: Dict[str, tuple] = {}
        for _ in range(p.itf8()):
            k = p.take(2).decode("ascii", "replace")
            self.series[k] = _parse_encoding(p)
        size = r.itf8()
        p = _Reader(r.take(size))
        self.tags: Dict[int, tuple] = {}
        for _ in range(p.itf8()):
            k = p.itf8()
            self.tags[k] = _parse_encoding(p)

    def program(self, cid_index: Dict[int, int]) -> np.ndarray:
        """The slice's int32 program (see include/unfazed_sm100.h) with content ids mapped to block indices."""
        encs: List[List[int]] = []
        pool: List[int] = []
        fixups = []                                  # (encoding number, position of a pool index)

        def add(e, i: Optional[int] = None) -> int:
            if i is None:
                i = len(encs)
                encs.append([0, 0, 0, 0])
            c = e[0]
            if c == E_EXTERNAL:
                encs[i] = [c, cid_index.get(e[1], -1), 0, 0]
            elif c == E_HUFFMAN:
                syms, lens = e[1], e[2]
                if len(syms) != len(lens) or not syms:
                    raise ValueError("HUFFMAN alphabet and code lengths differ in size")
                tab = canonical_codes(syms, lens)
                encs[i] = [c, len(tab), len(pool), 0]
                fixups.append(i)
                for code, ln, s in tab:
                    pool.extend([code, ln, s])
            elif c == E_BYTE_ARRAY_LEN:
                a = add(e[1])
                b = add(e[2])
                encs[i] = [c, a, b, 0]
            elif c == E_BYTE_ARRAY_STOP:
                encs[i] = [c, e[1], cid_index.get(e[2], -1), 0]
            elif c in (E_BETA, E_SUBEXP):
                encs[i] = [c, e[1], e[2], 0]
            elif c == E_GAMMA:
                encs[i] = [c, e[1], 0, 0]
            return i

        encs.extend([0, 0, 0, 0] for _ in SERIES)          # the data series first, at fixed numbers
        for i, s in enumerate(SERIES):
            add(self.series.get(s, (E_NULL,)), i)
        lines = []
        for line in self.td:
            lines.append([(k, add(self.tags[k]) if k in self.tags else _missing_tag(k)) for k in line])
        n = len(encs)
        base = 4 + 4 * n
        for i in fixups:
            encs[i][2] += base
        td = [len(lines)]
        off = 0
        for line in lines:
            td.append(off)
            off += len(line)
        td.append(off)
        for line in lines:
            for k, e in line:
                td += [k, e]
        prog = [n, base + len(pool), 0, 0] + [v for e in encs for v in e] + pool + td
        return np.array(prog, dtype=np.int32)


def _missing_tag(k: int) -> int:
    raise ValueError("tag %c%c:%c has no encoding" % (k >> 16, (k >> 8) & 0xFF, k & 0xFF))


def canonical_codes(syms: Sequence[int], lens: Sequence[int]) -> List[Tuple[int, int, int]]:
    """(code, length, symbol) of a canonical Huffman code, sorted by length then symbol (CRAM 3.0 section 13.4)."""
    order = sorted(zip(lens, syms))
    out, code, prev = [], 0, None
    for ln, s in order:
        if ln < 0 or ln > 31:
            raise ValueError("HUFFMAN code length %d out of range" % ln)
        if prev is not None:
            code = (code + 1) << (ln - prev)
        out.append((code, ln, s))
        prev = ln
    return out


class CramFile:
    """One CRAM 3.0 file with its CRAI index and a plain FASTA reference; with ``engine`` the slices are decoded on that
    engine's GPU."""

    def __init__(self, path: str, reference: Optional[str], index: Optional[str] = None, engine=None):
        self.path = path
        self.engine = engine
        self._containers: Dict[int, _Container] = {}
        with open(path, "rb") as f:
            size = os.fstat(f.fileno()).st_size
            self.data = mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ) if size else b""
        d = self.data
        if len(d) < 26 or d[:4] != b"CRAM":
            raise ValueError("%s: not a CRAM file (container offset 0)" % path)
        if (d[4], d[5]) != (3, 0):
            raise ValueError("%s: CRAM %d.%d is not read natively (container offset 0)" % (path, d[4], d[5]))
        eof_off = len(d) - len(EOF_CONTAINER)
        try:
            eof = self._container(eof_off) if eof_off >= 26 else None
        except ValueError:
            eof = None
        if eof is None or eof.ref_id != -1 or eof.start != EOF_START or eof.n_rec != 0:
            raise ValueError("%s: no CRAM EOF container at the end (container offset %d): truncated file?" % (path, max(eof_off, 0)))
        self.end = eof_off
        hc = self._container(26)
        blk = self._block(hc, hc.data_off)
        raw = self._block_data(hc, blk)
        if len(raw) < 4:
            raise ValueError("%s: empty SAM header block (container offset 26)" % path)
        ln = struct.unpack_from("<i", raw, 0)[0]
        self.text = raw[4:4 + ln].split(b"\0", 1)[0].decode("ascii", "replace")
        self.refs, self.ref_lens, rgs = [], [], []
        for line in self.text.splitlines():
            f = line.split("\t")
            kv = dict(x.split(":", 1) for x in f[1:] if ":" in x)
            if f[0] == "@SQ":
                self.refs.append(kv.get("SN", ""))
                self.ref_lens.append(int(kv.get("LN", "0")))
            elif f[0] == "@RG":
                rgs.append(kv.get("ID", ""))
        self.tids = {n: i for i, n in enumerate(self.refs)}
        self.read_groups = rgs
        tab = [b"RGZ" + g.encode() + b"\0" for g in rgs]
        offs = np.cumsum([0] + [len(t) for t in tab]) + 4 + 4 * (len(tab) + 1)
        self.rg_table = struct.pack("<i", len(tab)) + struct.pack("<%di" % len(offs), *offs.tolist()) + b"".join(tab)
        ip = index or index_path(path)
        if ip is None:
            raise ValueError("%s: no .crai index" % path)
        self.crai = self._read_crai(ip)
        self.reference = reference
        self._fasta: Optional[Fasta] = None

    # ---- low-level -------------------------------------------------------------------------------------------------
    def _err(self, off: int, msg: str) -> ValueError:
        return ValueError("%s: %s (container offset %d)" % (self.path, msg, off))

    def _container(self, off: int) -> _Container:
        c = self._containers.get(off)
        if c is not None:
            return c
        r = _Reader(self.data, off)
        try:
            c = _Container()
            c.off = off
            c.length = r.i32()
            c.ref_id, c.start, c.span, c.n_rec = r.itf8(), r.itf8(), r.itf8(), r.itf8()
            c.counter, _bases = r.ltf8(), r.ltf8()
            c.n_blocks = r.itf8()
            c.landmarks = r.itf8_array()
            crc_end = r.p
            crc = struct.unpack("<I", r.take(4))[0]
        except _Short:
            raise self._err(off, "truncated container header")
        if zlib.crc32(bytes(self.data[off:crc_end])) != crc:
            raise self._err(off, "container header fails its CRC32 check")
        c.data_off = r.p
        if c.length < 0 or c.data_off + c.length > len(self.data):
            raise self._err(off, "truncated container")
        c.comp = None
        self._containers[off] = c
        return c

    def _block(self, c: _Container, off: int) -> _Block:
        r = _Reader(self.data, off, c.data_off + c.length)
        b = _Block()
        try:
            b.method, b.ctype = r.byte(), r.byte()
            b.cid, b.size, b.raw_size = r.itf8(), r.itf8(), r.itf8()
            b.data_off = r.p
            r.take(b.size)
            crc = struct.unpack("<I", r.take(4))[0]
        except _Short:
            raise self._err(c.off, "truncated block at byte %d" % off)
        if zlib.crc32(bytes(self.data[off:b.data_off + b.size])) != crc:
            raise self._err(c.off, "block at byte %d fails its CRC32 check" % off)
        b.end = r.p
        return b

    def _block_data(self, c: _Container, b: _Block) -> bytes:
        try:
            return _decompress(b.method, bytes(self.data[b.data_off:b.data_off + b.size]), b.raw_size)
        except ValueError as e:
            raise self._err(c.off, str(e))
        except (OSError, EOFError, lzma.LZMAError, zlib.error) as e:
            raise self._err(c.off, "block does not decompress: %s" % e)

    def _comp(self, c: _Container) -> _CompHeader:
        if c.comp is None:
            b = self._block(c, c.data_off)
            if b.ctype != 1:
                raise self._err(c.off, "the first block is not a compression header")
            try:
                c.comp = _CompHeader(self._block_data(c, b))
            except _Short:
                raise self._err(c.off, "truncated compression header")
            except ValueError as e:
                raise self._err(c.off, str(e))
            if not c.comp.rn:
                raise self._err(c.off, "read names are not preserved (RN = false): mates cannot be joined")
        return c.comp

    def _read_crai(self, path: str) -> np.ndarray:
        try:
            text = gzip.decompress(open(path, "rb").read()).decode()
        except (OSError, EOFError):
            raise ValueError("%s: not a gzip-compressed CRAI index" % path)
        rows = [[int(x) for x in ln.split("\t")] for ln in text.splitlines() if ln.strip()]
        if any(len(r) != 6 for r in rows):
            raise ValueError("%s: a CRAI line does not have 6 fields" % path)
        a = np.array(rows, dtype=np.int64).reshape(-1, 6)
        return a

    def fasta(self) -> Fasta:
        if self._fasta is None:
            if not self.reference:
                raise ValueError("%s: a reference (-r) is needed to decode this CRAM" % self.path)
            self._fasta = Fasta(self.reference)
        return self._fasta

    # ---- queries -----------------------------------------------------------------------------------------------------
    def slices_for(self, queries: Sequence[Tuple[int, int, int]]) -> List[Tuple[int, int]]:
        """(container offset, slice offset) of every slice overlapping a (tid, beg, end) query, once, in file order."""
        a = self.crai
        keep = np.zeros(a.shape[0], dtype=bool)
        for tid, beg, end in queries:
            end = max(end, beg + 1)
            keep |= (a[:, 0] == tid) & (a[:, 1] - 1 < end) & (a[:, 1] - 1 + a[:, 2] > beg)
        return sorted(set(zip(a[keep, 3].tolist(), a[keep, 4].tolist())))

    def fetch_union(self, queries: Sequence[Tuple[int, int, int]]) -> Tuple[np.ndarray, np.ndarray]:
        """BAM record bytes and record offsets of every slice overlapping one of the (tid, beg, end) queries; a slice
        shared by several queries is decoded once.  Selection is the caller's."""
        return self.decode(self.slices_for(queries))

    def head_tlen(self, n: int) -> np.ndarray:
        """Template lengths of the first n records of the file."""
        if n <= 0:
            return np.zeros(0, dtype=np.int64)
        allsl = sorted(set(zip(self.crai[:, 3].tolist(), self.crai[:, 4].tolist())))
        out: List[np.ndarray] = []
        got, i = 0, 0
        while got < n and i < len(allsl):
            step = allsl[i:i + 4]
            i += 4
            buf, offs = self.decode(step, engine=False)
            offs = offs[: n - got]
            out.append(buf[offs[:, None] + np.arange(32, 36)].copy().view("<i4").reshape(-1).astype(np.int64))
            got += offs.shape[0]
        return np.concatenate(out) if out else np.zeros(0, dtype=np.int64)

    # ---- decode ------------------------------------------------------------------------------------------------------
    def prepare(self, slices: Sequence[Tuple[int, int]]):
        """The flat descriptors of these slices: (slices, blocks, ext, prog, refs, rbytes, n_records, container offsets)."""
        heads = []                                    # (container, slice header, [blocks])
        for coff, soff in slices:
            c = self._container(coff)
            comp = self._comp(c)
            p = c.data_off + soff
            hb = self._block(c, p)
            if hb.ctype != 2:
                raise self._err(coff, "no slice header at landmark %d" % soff)
            try:
                r = _Reader(self._block_data(c, hb))
                sh = dict(ref_id=r.itf8(), start=r.itf8(), span=r.itf8(), n_rec=r.itf8(), counter=r.ltf8())
                n_blocks = r.itf8()
                sh["cids"] = r.itf8_array()
                sh["emb"] = r.itf8()
                sh["md5"] = r.take(16)
            except _Short:
                raise self._err(coff, "truncated slice header")
            blocks, q = [], hb.end
            for _ in range(n_blocks):
                b = self._block(c, q)
                blocks.append(b)
                q = b.end
            heads.append((c, comp, sh, blocks))
        # every block of every slice decompressed in the thread pool
        jobs = [(c, b) for c, _comp, _sh, bl in heads for b in bl]
        with ThreadPoolExecutor(_THREADS) as ex:
            datas = list(ex.map(lambda cb: self._block_data(*cb), jobs)) if len(jobs) > 1 else \
                [self._block_data(*cb) for cb in jobs]
        parts: List[bytes] = [self.rg_table]
        size = len(self.rg_table)
        sl = np.zeros(len(heads), dtype=SLICE_DTYPE)
        exts, progs, refs, rparts = [], [], [], []
        prog_size, rsize, rec = 0, 0, 0
        ref_cache: Dict[Tuple[int, int, int], int] = {}
        k = 0
        for si, (c, comp, sh, bl) in enumerate(heads):
            core = None
            ext_of: Dict[int, int] = {}
            slice_ext = []
            emb = None
            for b in bl:
                data = datas[k]
                k += 1
                off = size
                parts.append(data)
                size += len(data)
                if b.ctype == 5:
                    core = (off, len(data))
                elif b.ctype == 4:
                    ext_of[b.cid] = len(slice_ext)
                    slice_ext.append((off, len(data)))
                    if b.cid == sh["emb"]:
                        emb = data
            if core is None:
                raise self._err(c.off, "slice without a core data block")
            if len(slice_ext) > L.CRAM_MAX_EXT:
                raise self._err(c.off, "more than %d external blocks in a slice" % L.CRAM_MAX_EXT)
            try:
                prog = comp.program(ext_of)
            except ValueError as e:
                raise self._err(c.off, str(e))
            s = sl[si]
            s["core_off"], s["core_len"] = core
            s["ext_off"], s["n_ext"] = len(exts), len(slice_ext)
            exts += slice_ext
            s["prog_off"] = prog_size
            progs.append(prog)
            prog_size += prog.shape[0]
            s["rec_first"], s["n_records"] = rec, sh["n_rec"]
            rec += sh["n_rec"]
            s["rg_off"] = 0
            s["ref_id"], s["ap_start"] = sh["ref_id"], sh["start"]
            s["flags"] = AP_DELTA if comp.ap_delta else 0
            s["sub"] = np.frombuffer(comp.sub, dtype=np.uint8)
            # reference spans
            spans = []
            if comp.rr and sh["ref_id"] >= 0 and emb is None:
                name = self._ref_name(c, sh["ref_id"])
                beg, end = sh["start"] - 1, sh["start"] - 1 + sh["span"]
                key = (sh["ref_id"], beg, end)
                if key not in ref_cache:
                    seq = self.fasta().fetch(name, beg, end)
                    if sh["md5"] != bytes(16) and hashlib.md5(seq).digest() != sh["md5"]:
                        raise self._err(c.off, "slice MD5 does not match reference %s:%d-%d" % (name, beg + 1, end))
                    ref_cache[key] = len(refs)
                    refs.append((rsize, beg, len(seq), sh["ref_id"]))
                    rparts.append(seq)
                    rsize += len(seq)
                spans = [ref_cache[key]]
            elif emb is not None and sh["ref_id"] >= 0:
                spans = [len(refs)]
                refs.append((rsize, sh["start"] - 1, len(emb), sh["ref_id"]))
                rparts.append(emb)
                rsize += len(emb)
            elif comp.rr and sh["ref_id"] == -2:
                for t, name in enumerate(self.refs):
                    key = (t, 0, -1)
                    if key not in ref_cache:
                        seq = self.fasta().fetch(name, 0, self.fasta().length(name)) if name in self.fasta().index else b""
                        ref_cache[key] = len(refs)
                        refs.append((rsize, 0, len(seq), t))
                        rparts.append(seq)
                        rsize += len(seq)
                    spans.append(ref_cache[key])
            # the slice's spans are consecutive entries: copy them behind the others when they are not
            if spans and spans != list(range(spans[0], spans[0] + len(spans))):
                first = len(refs)
                refs += [refs[j] for j in spans]
                spans = list(range(first, first + len(spans)))
            s["refs_off"] = spans[0] if spans else 0
            s["n_refs"] = len(spans)
        blocks = np.frombuffer(b"".join(parts), dtype=np.uint8) if size else np.zeros(1, dtype=np.uint8)
        ext = np.array(exts, dtype=np.int64).reshape(-1, 2).copy().view(EXT_DTYPE).reshape(-1) if exts else \
            np.zeros(1, dtype=EXT_DTYPE)
        prog = np.concatenate(progs) if progs else np.zeros(1, dtype=np.int32)
        ref = np.zeros(max(len(refs), 1), dtype=REF_DTYPE)
        for j, (o, st, ln, t) in enumerate(refs):
            ref[j]["off"], ref[j]["start"], ref[j]["len"], ref[j]["ref_id"] = o, st, ln, t
        rbytes = np.frombuffer(b"".join(rparts), dtype=np.uint8) if rsize else np.zeros(1, dtype=np.uint8)
        return sl, blocks, ext, prog, ref, rbytes, rec, [h[0].off for h in heads]

    def _ref_name(self, c: _Container, tid: int) -> str:
        if tid >= len(self.refs):
            raise self._err(c.off, "reference id %d is not in the header" % tid)
        name = self.refs[tid]
        if name not in self.fasta().index:
            raise self._err(c.off, "reference %s is not in %s" % (name, self.reference))
        return name

    def decode(self, slices: Sequence[Tuple[int, int]], engine=None) -> Tuple[np.ndarray, np.ndarray]:
        """BAM record bytes and offsets of these slices (host entry points, or the engine's GPU)."""
        if not slices:
            return np.zeros(0, dtype=np.uint8), np.zeros(0, dtype=np.int64)
        desc = self.prepare(slices)
        eng = self.engine if engine is None else (engine or None)
        if eng is not None:
            return eng.cram_decoder().decode(self, desc)
        sl, blocks, ext, prog, ref, rbytes, n_rec, coffs = desc
        lib = L.load()
        rec_len = np.zeros(max(n_rec, 1), dtype=np.int64)
        rec_cig = np.zeros(max(n_rec, 1), dtype=np.int32)
        status = np.zeros(sl.shape[0], dtype=np.int32)
        args = (_ptr(sl), int(sl.shape[0]), _ptr(blocks), _ptr(ext), _ptr(prog), _ptr(ref), _ptr(rbytes))
        lib.unfz_cram_decode_size_host(*args, _ptr(rec_len), _ptr(rec_cig), _ptr(status))
        self.check_status(status, coffs)
        offs = np.zeros(n_rec + 1, dtype=np.int64)
        np.cumsum(rec_len[:n_rec], out=offs[1:])
        out = np.zeros(max(int(offs[-1]), 1), dtype=np.uint8)
        lib.unfz_cram_decode_write_host(*args, _ptr(rec_cig), _ptr(offs), _ptr(out), _ptr(status))
        self.check_status(status, coffs)
        return out[: int(offs[-1])], offs[:-1].copy()

    def check_status(self, status: np.ndarray, coffs: Sequence[int]) -> None:
        bad = np.flatnonzero(status)
        if bad.shape[0]:
            i = int(bad[0])
            raise self._err(coffs[i], "slice does not decode: %s" % STATUS.get(int(status[i]), "status %d" % status[i]))


def is_native_cram(path: str, reference: Optional[str]) -> bool:
    """An existing CRAM 3.0 file with a ``.crai`` and a plain-text FASTA reference: read by ``CramFile``."""
    return (path.endswith(".cram") and os.path.isfile(path) and file_version(path) == (3, 0)
            and index_path(path) is not None and is_plain_fasta(reference))


# ------------------------------------------------------------------------------------------------
# writer
# ------------------------------------------------------------------------------------------------

class _Bits:
    def __init__(self):
        self.out = bytearray()
        self.cur = 0
        self.n = 0

    def put(self, v: int, nbits: int):
        for i in range(nbits - 1, -1, -1):
            self.cur = (self.cur << 1) | ((v >> i) & 1)
            self.n += 1
            if self.n == 8:
                self.out.append(self.cur)
                self.cur = self.n = 0

    def bytes(self) -> bytes:
        return bytes(self.out) + (bytes([self.cur << (8 - self.n)]) if self.n else b"")


def huffman_lengths(freq: Dict[int, int]) -> Dict[int, int]:
    """Code lengths of a Huffman code for these symbol counts (one symbol: length 0)."""
    if len(freq) == 1:
        return {next(iter(freq)): 0}
    heap = [(f, i, [s]) for i, (s, f) in enumerate(sorted(freq.items()))]
    heapq.heapify(heap)
    depth = {s: 0 for s in freq}
    cnt = len(heap)
    while len(heap) > 1:
        f1, _, a = heapq.heappop(heap)
        f2, _, b = heapq.heappop(heap)
        for s in a + b:
            depth[s] += 1
        heapq.heappush(heap, (f1 + f2, cnt, a + b))
        cnt += 1
    return depth


def _enc_bytes(e: tuple) -> bytes:
    c = e[0]
    if c == E_EXTERNAL:
        p = itf8(e[1])
    elif c == E_HUFFMAN:
        p = itf8(len(e[1])) + b"".join(itf8(x) for x in e[1]) + itf8(len(e[2])) + b"".join(itf8(x) for x in e[2])
    elif c == E_BYTE_ARRAY_LEN:
        p = _enc_bytes(e[1]) + _enc_bytes(e[2])
    elif c == E_BYTE_ARRAY_STOP:
        p = bytes([e[1]]) + itf8(e[2])
    elif c in (E_BETA, E_SUBEXP, E_GOLOMB, E_GOLOMB_RICE):
        p = itf8(e[1]) + itf8(e[2])
    elif c == E_GAMMA:
        p = itf8(e[1])
    else:
        p = b""
    return itf8(c) + itf8(len(p)) + p


def _core_encoding(series: str, vals: List[int]) -> tuple:
    """The bit-stream encoding the writer's ``encoding="core"`` gives a series, from its values."""
    if not vals:
        return (E_NULL,)
    lo, hi = min(vals), max(vals)
    if series in ("BF", "CF", "MQ", "FC", "BS", "TL", "RG", "MF", "RI", "QS"):
        freq: Dict[int, int] = {}
        for v in vals:
            freq[v] = freq.get(v, 0) + 1
        ln = huffman_lengths(freq)
        syms = sorted(ln)
        return (E_HUFFMAN, syms, [ln[s] for s in syms])
    if series in ("RL", "FN", "NF"):
        return (E_BETA, -lo, max(1, (hi - lo).bit_length()))
    if series in ("FP", "DL", "HC", "PD", "RS"):
        return (E_GAMMA, 1 - lo)
    if series == "AP":
        return (E_SUBEXP, -lo, 2)
    return None


def write_cram(table, kid: int, path: str, reference: str, method="gzip", encoding="external", records_per_slice=10000,
               slices_per_container=1, multi_ref=False, embed_ref=False, rr=True, **bam_opts) -> None:
    """Coordinate-sorted CRAM 3.0 + ``path + ".crai"`` of kid ``kid``'s reads of ``table``, against the plain FASTA
    ``reference``.  The records are those ``bamio.write_bam`` writes with the same ``bam_opts`` (tags, missing
    qualities, mates on other references), so the two files decode to the same BAM records.

    ``method``: the block method (raw, gzip, bzip2, lzma, rans0, rans1) of every block, or a dict by data series / tag
    key (``"*"`` the default).  ``encoding``: "external" (every series in its own external block) or "core" (HUFFMAN,
    BETA, GAMMA and SUBEXP in the core bit stream where they fit, BYTE_ARRAY_STOP for names and strings), or a dict of
    series -> encoding tuple overriding either.  ``multi_ref``: slices mix references (RI per record).  ``embed_ref``:
    every slice carries its reference span.  ``rr`` False: no reference is needed to decode (every base is stored)."""
    with tempfile.TemporaryDirectory() as td:
        bp = os.path.join(td, "r.bam")
        bamio.write_bam(table, kid, bp, **bam_opts)
        bf = bamio.BamFile(bp)
        buf, _ = bf.bgzf.stream_from(bf.first_voff, 1 << 62)
        offs, _ = bamio.record_offsets(buf)
        refs, ref_lens, text = bf.refs, bf.ref_lens, bf.text
    recs = [_bam_fields(buf, int(o)) for o in offs.tolist()]
    fa = Fasta(reference)
    rgs: List[str] = []
    for r in recs:
        g = r["rg"]
        if g is not None and g not in rgs:
            rgs.append(g)
    text = text + "".join("@RG\tID:%s\n" % g for g in rgs)
    write_cram_records(recs, path, refs, ref_lens, text, fa, method=method, encoding=encoding,
                       records_per_slice=records_per_slice, slices_per_container=slices_per_container,
                       multi_ref=multi_ref, embed_ref=embed_ref, rr=rr)


def _bam_fields(buf: np.ndarray, o: int) -> dict:
    b = buf[o: o + 4 + int(buf[o:o + 4].view("<i4")[0])].tobytes()
    bs, rid, pos, ln, mq, _bin, nc, flag, ls, nrid, npos, tlen = struct.unpack_from("<iiiBBHHHiiii", b, 0)
    p = 36
    name = b[p:p + ln - 1]
    p += ln
    cig = list(struct.unpack_from("<%dI" % nc, b, p))
    p += 4 * nc
    sb = (ls + 1) // 2
    nib = "=ACMGRSVTWYHKDBN"
    seq = "".join(nib[(b[p + k // 2] >> (0 if k & 1 else 4)) & 15] for k in range(ls)).encode()
    p += sb
    qual = b[p:p + ls]
    p += ls
    aux = b[p:]
    # aux fields split into (key, value bytes); RG:Z moves to the RG series when it is the last field
    tags, q = [], 0
    while q < len(aux):
        t = aux[q:q + 3]
        n = _aux_len(aux, q + 3, t[2:3])
        tags.append(((t[0] << 16) | (t[1] << 8) | t[2], aux[q + 3:q + 3 + n]))
        q += 3 + n
    rg = None
    if tags and tags[-1][0] == (ord("R") << 16) | (ord("G") << 8) | ord("Z"):
        rg = tags[-1][1][:-1].decode()
        tags = tags[:-1]
    return dict(rid=rid, pos=pos, mapq=mq, cigar=cig, flag=flag, seq=seq, qual=qual, name=name, tags=tags, rg=rg,
                nrid=nrid, npos=npos, tlen=tlen, missing=ls > 0 and qual[:1] == b"\xff")


def _aux_len(aux: bytes, p: int, t: bytes) -> int:
    t = t.decode()
    if t in "AcC":
        return 1
    if t in "sS":
        return 2
    if t in "iIf":
        return 4
    if t in "ZH":
        return aux.index(b"\0", p) - p + 1
    if t == "B":
        sub = chr(aux[p])
        cnt = struct.unpack_from("<I", aux, p + 1)[0]
        return 5 + cnt * {"c": 1, "C": 1, "s": 2, "S": 2, "i": 4, "I": 4, "f": 4}[sub]
    raise ValueError("unknown aux type %r" % t)


def _ref_len(cig: List[int]) -> int:
    return sum(w >> 4 for w in cig if (w & 15) in (0, 2, 3, 7, 8))


def _features(r: dict, ref: bytes, ref_beg: int, rr: bool, sub_code) -> Tuple[list, List[int]]:
    """The read features of a mapped record and the CIGAR the decoder rebuilds from them."""
    feats = []
    rp, gp = 0, r["pos"]
    seq, missing = r["seq"], r["missing"]
    for w in r["cigar"]:
        op, n = w & 15, w >> 4
        if op in (0, 7, 8):
            if not rr:
                feats.append((rp + 1, "b", seq[rp:rp + n]))
            else:
                for k in range(n):
                    rb = seq[rp + k]
                    fb = ref[gp + k - ref_beg] if 0 <= gp + k - ref_beg < len(ref) else ord("N")
                    if rb == fb:
                        continue
                    if rb in b"ACGTN" and fb != rb and sub_code(fb, rb) is not None:
                        feats.append((rp + k + 1, "X", sub_code(fb, rb)))
                    elif missing:
                        feats.append((rp + k + 1, "b", bytes([rb])))
                    else:
                        feats.append((rp + k + 1, "B", (rb, r["qual"][rp + k])))
            rp += n
            gp += n
        elif op == 1:
            feats.append((rp + 1, "i", seq[rp]) if n == 1 else (rp + 1, "I", seq[rp:rp + n]))
            rp += n
        elif op == 4:
            feats.append((rp + 1, "S", seq[rp:rp + n]))
            rp += n
        elif op == 2:
            feats.append((rp + 1, "D", n))
            gp += n
        elif op == 3:
            feats.append((rp + 1, "N", n))
            gp += n
        elif op == 6:
            feats.append((rp + 1, "P", n))
        elif op == 5:
            feats.append((rp + 1, "H", n))
        else:
            raise ValueError("CIGAR operation %d cannot be stored in CRAM" % op)
    # the CIGAR the decoder rebuilds: runs of the same operation merged, matches and mismatches as M
    rebuilt: List[List[int]] = []

    def add(op, n):
        if n <= 0:
            return
        if rebuilt and rebuilt[-1][0] == op:
            rebuilt[-1][1] += n
        else:
            rebuilt.append([op, n])
    pos = 0
    opmap = {"i": 1, "I": 1, "S": 4, "D": 2, "N": 3, "P": 6, "H": 5}
    for fp, fc, v in feats:
        add(0, fp - 1 - pos)
        pos = max(pos, fp - 1)
        if fc in "XB":
            add(0, 1)
            pos += 1
        elif fc == "b":
            add(0, len(v))
            pos += len(v)
        elif fc in "IS":
            add(opmap[fc], len(v))
            pos += len(v)
        elif fc == "i":
            add(1, 1)
            pos += 1
        else:
            add(opmap[fc], v)
    add(0, len(seq) - pos)
    return feats, [(n << 4) | op for op, n in rebuilt]


def write_cram_records(recs: List[dict], path: str, refs: List[str], ref_lens: List[int], text: str, fa: Fasta,
                       method="gzip", encoding="external", records_per_slice=10000, slices_per_container=1,
                       multi_ref=False, embed_ref=False, rr=True) -> None:
    """The CRAM writer behind ``write_cram``, from records in BAM field form (``_bam_fields``)."""
    sub = bytes([0x1B, 0x1B, 0x1B, 0x1B, 0x1B])   # codes 0..3 for the other bases in ACGTN order
    letters = b"ACGTN"

    def sub_code(fb, rb):
        r = letters.find(bytes([fb])) if bytes([fb]) in letters else 4
        alts = [x for x in letters if x != letters[r]]
        return alts.index(rb) if rb in alts else None
    rg_index = {}
    for line in text.splitlines():
        if line.startswith("@RG"):
            kv = dict(x.split(":", 1) for x in line.split("\t")[1:] if ":" in x)
            rg_index[kv["ID"]] = len(rg_index)
    # ---- slices: runs of records of one reference (or mixed with multi_ref) ----------------------------------------
    groups: List[List[int]] = []
    for i, r in enumerate(recs):
        if groups and len(groups[-1]) < records_per_slice and (multi_ref or recs[groups[-1][0]]["rid"] == r["rid"]):
            groups[-1].append(i)
        else:
            groups.append([i])
    ap_delta = not multi_ref
    header_raw = struct.pack("<i", len(text)) + text.encode()
    out = bytearray(b"CRAM\x03\x00" + os.path.basename(path).encode()[:20].ljust(20, b"\0"))
    out += container_bytes(0, 0, 0, 0, 0, 0, 1, [0], block_bytes(0, 0, 0, len(header_raw), header_raw))
    crai: List[Tuple[int, int, int, int, int, int]] = []
    counter = 0
    whole: Dict[int, bytes] = {}                       # whole reference sequences of multi-reference slices
    meth = method if isinstance(method, dict) else {"*": method}
    enc_over = encoding if isinstance(encoding, dict) else {}
    core_mode = encoding == "core" or (isinstance(encoding, dict) and encoding.get("*") == "core")
    # content ids: series i -> 11 + i; BYTE_ARRAY_LEN lengths -> 51 + i; tags from 100; the embedded reference 9999
    for c0 in range(0, len(groups), slices_per_container):
        cgroups = groups[c0:c0 + slices_per_container]
        # ---- per-slice record values -----------------------------------------------------------------------------------
        slice_vals = []
        td_lines: List[Tuple[int, ...]] = []
        td_index: Dict[Tuple[int, ...], int] = {}
        tag_keys: Dict[int, str] = {}
        for g in cgroups:
            rs = [recs[i] for i in g]
            rids = sorted({r["rid"] for r in rs})
            sref = rids[0] if len(rids) == 1 else -2
            mapped = [r for r in rs if r["pos"] >= 0]
            if sref >= 0 and mapped:
                sstart = min(r["pos"] for r in mapped) + 1
                send = max(r["pos"] + max(_ref_len(r["cigar"]), 1) for r in mapped)
            else:
                sstart, send = 0, 0
            ref = fa.fetch(refs[sref], sstart - 1, send) if sref >= 0 and sstart > 0 else b""
            V = {s: [] for s in SERIES}
            T: Dict[int, list] = {}
            mates = _mate_plan(rs)
            prev = sstart
            for j, r in enumerate(rs):
                flag = r["flag"]
                kind, nf = mates[j]
                cf = (0 if r["missing"] or not r["seq"] else 1) | (8 if not r["seq"] else 0)
                if kind == "detached":
                    cf |= 2
                    flag &= ~0x28
                elif kind == "attached":
                    cf |= 4
                    flag &= ~0x28
                elif kind == "last":
                    flag &= ~0x28
                V["BF"].append(flag)
                V["CF"].append(cf)
                if sref == -2:
                    V["RI"].append(r["rid"])
                V["RL"].append(len(r["seq"]))
                ap = r["pos"] + 1
                V["AP"].append(ap - prev if ap_delta else ap)
                if ap_delta:
                    prev = ap
                V["RG"].append(rg_index[r["rg"]] if r["rg"] is not None else -1)
                V["RN"].append(r["name"])
                if kind == "detached":
                    V["MF"].append((1 if r["flag"] & 0x20 else 0) | (2 if r["flag"] & 0x8 else 0))
                    V["NS"].append(r["nrid"])
                    V["NP"].append(r["npos"] + 1)
                    V["TS"].append(r["tlen"])
                elif kind == "attached":
                    V["NF"].append(nf)
                line = tuple(k for k, _v in r["tags"])
                if line not in td_index:
                    td_index[line] = len(td_lines)
                    td_lines.append(line)
                V["TL"].append(td_index[line])
                for k, v in r["tags"]:
                    T.setdefault(k, []).append(v)
                    tag_keys[k] = ""
                if not r["flag"] & 0x4:
                    if not r["seq"] and any((w & 15) in (0, 1, 4, 7, 8) for w in r["cigar"]):
                        raise ValueError("a mapped record without bases but with a query-consuming CIGAR is not written")
                    if sref == -2:
                        if r["rid"] not in whole:
                            name = refs[r["rid"]]
                            whole[r["rid"]] = fa.fetch(name, 0, fa.length(name)) if name in fa.index else b""
                        feats, rebuilt = _features(r, whole[r["rid"]], 0, rr, sub_code)
                    else:
                        feats, rebuilt = _features(r, ref, sstart - 1, rr, sub_code)
                    if rebuilt != r["cigar"]:
                        raise ValueError("record %r: CIGAR %r cannot be rebuilt from CRAM features" % (r["name"], r["cigar"]))
                    V["FN"].append(len(feats))
                    last = 0
                    for fp, fc, v in feats:
                        V["FC"].append(ord(fc))
                        V["FP"].append(fp - last)
                        last = fp
                        if fc == "X":
                            V["BS"].append(v)
                        elif fc == "B":
                            V["BA"].append(v[0])
                            V["QS"].append(v[1])
                        elif fc == "i":
                            V["BA"].append(v)
                        elif fc == "I":
                            V["IN"].append(v)
                        elif fc == "S":
                            V["SC"].append(v)
                        elif fc == "b":
                            V["BB"].append(v)
                        elif fc == "D":
                            V["DL"].append(v)
                        elif fc == "N":
                            V["RS"].append(v)
                        elif fc == "P":
                            V["PD"].append(v)
                        elif fc == "H":
                            V["HC"].append(v)
                    V["MQ"].append(r["mapq"])
                else:
                    if r["cigar"] or r["mapq"]:
                        raise ValueError("record %r: an unmapped record with a CIGAR or MAPQ is not written" % r["name"])
                    V["BA"].extend(r["seq"])
                if cf & 1:
                    V["QS"].extend(r["qual"])
            slice_vals.append((sref, sstart, send, rs, V, T, ref))
        # ---- encodings of this container ----------------------------------------------------------------------------
        allv = {s: [v for sv in slice_vals for v in sv[4][s]] for s in SERIES}
        encs: Dict[str, tuple] = {}
        for i, s in enumerate(SERIES):
            e = None
            if s in enc_over:
                e = enc_over[s]
            elif core_mode and s not in _ARRAY_SERIES:
                e = _core_encoding(s, allv[s])
            elif core_mode and s in ("RN", "IN", "SC"):
                e = (E_BYTE_ARRAY_STOP, 0, 11 + i)
            if e is None:
                if s in _ARRAY_SERIES:
                    e = (E_BYTE_ARRAY_LEN, (E_EXTERNAL, 51 + i), (E_EXTERNAL, 11 + i))
                else:
                    e = (E_EXTERNAL, 11 + i)
            encs[s] = e
        tag_enc: Dict[int, tuple] = {}
        for j, k in enumerate(sorted(tag_keys)):
            typ = chr(k & 0xFF)
            vals = [v for sv in slice_vals for v in sv[5].get(k, [])]
            if core_mode and typ in "ZH" and all(b"\t" not in v[:-1] for v in vals):
                tag_enc[k] = (E_BYTE_ARRAY_STOP, 9, 100 + 2 * j)
            else:
                tag_enc[k] = (E_BYTE_ARRAY_LEN, (E_EXTERNAL, 101 + 2 * j), (E_EXTERNAL, 100 + 2 * j))
        # ---- compression header ---------------------------------------------------------------------------------------
        td_raw = b"".join(b"".join(bytes([(k >> 16) & 0xFF, (k >> 8) & 0xFF, k & 0xFF]) for k in line) + b"\0"
                          for line in (td_lines or [()]))
        pm = [b"RN\x01", b"AP" + bytes([ap_delta]), b"RR" + bytes([rr]), b"SM" + sub, b"TD" + itf8(len(td_raw)) + td_raw]
        pm_raw = itf8(len(pm)) + b"".join(pm)
        used = [s for s in SERIES if allv[s] or s in ("BF", "CF", "RL", "AP", "RG", "RN", "TL", "MQ", "FN")]
        ds_raw = itf8(len(used)) + b"".join(s.encode() + _enc_bytes(encs[s]) for s in used)
        te_raw = itf8(len(tag_enc)) + b"".join(itf8(k) + _enc_bytes(e) for k, e in sorted(tag_enc.items()))
        comp_raw = itf8(len(pm_raw)) + pm_raw + itf8(len(ds_raw)) + ds_raw + itf8(len(te_raw)) + te_raw
        body = bytearray(block_bytes(0, 1, 0, len(comp_raw), comp_raw))
        landmarks = []
        n_blocks = 1
        c_bases = 0
        slice_info = []
        for sref, sstart, send, rs, V, T, ref in slice_vals:
            streams: Dict[int, bytearray] = {}
            bits = _Bits()
            huff: Dict[tuple, dict] = {}

            def put(e, v, is_byte, s=None):
                c = e[0]
                if c == E_EXTERNAL:
                    streams.setdefault(e[1], bytearray()).extend(bytes([v & 0xFF]) if is_byte else itf8(v))
                elif c == E_HUFFMAN:
                    key = (tuple(e[1]), tuple(e[2]))
                    if key not in huff:
                        huff[key] = {sym: (code, ln) for code, ln, sym in canonical_codes(e[1], e[2])}
                    code, ln = huff[key][v]
                    bits.put(code, ln)
                elif c == E_BETA:
                    bits.put(v + e[1], e[2])
                elif c == E_GAMMA:
                    x = v + e[1]
                    nb = x.bit_length() - 1
                    bits.put(0, nb)
                    bits.put(x, nb + 1)
                elif c == E_SUBEXP:
                    x, k = v + e[1], e[2]
                    if x < (1 << k):
                        bits.put(0, 1)
                        bits.put(x, k)
                    else:
                        b = x.bit_length() - 1
                        u = b - k + 1
                        bits.put((1 << u) - 1, u)
                        bits.put(0, 1)
                        bits.put(x - (1 << b), b)
                elif c != E_NULL:
                    raise ValueError("encoding %d cannot hold a single value" % c)

            def put_array(e, v: bytes):
                if e[0] == E_BYTE_ARRAY_LEN:
                    put(e[1], len(v), False)
                    for x in v:
                        put(e[2], x, True)
                elif e[0] == E_BYTE_ARRAY_STOP:
                    streams.setdefault(e[2], bytearray()).extend(bytes(v) + bytes([e[1]]))
                else:
                    raise ValueError("encoding %d cannot hold a byte array" % e[0])
            # values in decode order, record by record
            cursors = {s: 0 for s in SERIES}
            tcur = {k: 0 for k in T}

            def nxt(s):
                v = V[s][cursors[s]]
                cursors[s] += 1
                return v
            for j, r in enumerate(rs):
                for s in ("BF", "CF") + (("RI",) if sref == -2 else ()) + ("RL", "AP", "RG"):
                    put(encs[s], nxt(s), False)
                put_array(encs["RN"], nxt("RN"))
                cf = V["CF"][j]
                if cf & 2:
                    for s in ("MF", "NS", "NP", "TS"):
                        put(encs[s], nxt(s), False)
                elif cf & 4:
                    put(encs["NF"], nxt("NF"), False)
                put(encs["TL"], nxt("TL"), False)
                for k, _v in r["tags"]:
                    v = T[k][tcur[k]]
                    tcur[k] += 1
                    e = tag_enc[k]
                    put_array(e, v[:-1] if e[0] == E_BYTE_ARRAY_STOP else v)
                if not r["flag"] & 0x4:
                    fn = nxt("FN")
                    put(encs["FN"], fn, False)
                    for _ in range(fn):
                        fc = nxt("FC")
                        put(encs["FC"], fc, True)
                        put(encs["FP"], nxt("FP"), False)
                        fc = chr(fc)
                        if fc == "X":
                            put(encs["BS"], nxt("BS"), True)
                        elif fc == "B":
                            put(encs["BA"], nxt("BA"), True)
                            put(encs["QS"], nxt("QS"), True)
                        elif fc == "i":
                            put(encs["BA"], nxt("BA"), True)
                        elif fc in "ISb":
                            s = {"I": "IN", "S": "SC", "b": "BB"}[fc]
                            put_array(encs[s], nxt(s))
                        else:
                            s = {"D": "DL", "N": "RS", "P": "PD", "H": "HC"}[fc]
                            put(encs[s], nxt(s), False)
                    put(encs["MQ"], nxt("MQ"), False)
                else:
                    for _ in range(len(r["seq"])):
                        put(encs["BA"], nxt("BA"), True)
                if cf & 1:
                    for _ in range(len(r["seq"])):
                        put(encs["QS"], nxt("QS"), True)
            emb_id = -1
            if embed_ref and sref >= 0 and ref:
                emb_id = 9999
                streams[emb_id] = bytearray(ref)
            blocks = [block_bytes(0, 5, 0, len(bits.bytes()), bits.bytes())]
            cids = []
            for cid in sorted(streams):
                raw = bytes(streams[cid])
                key = next((s for i, s in enumerate(SERIES) if cid in (11 + i, 51 + i)), None)
                m = meth.get(key, meth.get("*", "gzip")) if key else meth.get(cid, meth.get("*", "gzip"))
                mid, data = _compress(raw, m)
                blocks.append(block_bytes(mid, 4, cid, len(raw), data))
                cids.append(cid)
            md5 = hashlib.md5(ref).digest() if (sref >= 0 and rr and ref) else bytes(16)
            counter_s = counter
            counter += len(rs)
            sh = (itf8(sref) + itf8(sstart) + itf8(send - sstart + 1 if sstart else 0) + itf8(len(rs)) + ltf8(counter_s)
                  + itf8(len(blocks)) + itf8(len(cids) + 1) + itf8(0) + b"".join(itf8(c) for c in cids) + itf8(emb_id) + md5)
            landmarks.append(len(body))
            sbytes = block_bytes(0, 2, 0, len(sh), sh) + b"".join(blocks)
            body += sbytes
            n_blocks += 1 + len(blocks)
            c_bases += sum(len(r["seq"]) for r in rs)
            slice_info.append((sref, sstart, send, rs, landmarks[-1], len(sbytes)))
        refs_c = {si[0] for si in slice_info}
        cref = next(iter(refs_c)) if len(refs_c) == 1 else -2
        cstart = min((si[1] for si in slice_info if si[1]), default=0)
        cend = max((si[2] for si in slice_info), default=0)
        coff = len(out)
        out += container_bytes(cref, cstart if cref >= 0 else 0, (cend - cstart + 1) if cref >= 0 and cstart else 0,
                               sum(len(si[3]) for si in slice_info), counter - sum(len(si[3]) for si in slice_info),
                               c_bases, n_blocks, landmarks, bytes(body))
        for sref, sstart, send, rs, soff, ssize in slice_info:
            if sref == -2:
                for t in sorted({r["rid"] for r in rs}):
                    m = [r for r in rs if r["rid"] == t and r["pos"] >= 0]
                    if t >= 0 and m:
                        a = min(r["pos"] for r in m) + 1
                        b = max(r["pos"] + max(_ref_len(r["cigar"]), 1) for r in m)
                        crai.append((t, a, b - a + 1, coff, soff, ssize))
                    else:
                        crai.append((-1, 0, 0, coff, soff, ssize))
            elif sref >= 0 and sstart:
                crai.append((sref, sstart, send - sstart + 1, coff, soff, ssize))
            else:
                crai.append((-1, 0, 0, coff, soff, ssize))
    out += EOF_CONTAINER
    with open(path, "wb") as f:
        f.write(bytes(out))
    with open(path + ".crai", "wb") as f:
        f.write(gzip.compress("".join("%d\t%d\t%d\t%d\t%d\t%d\n" % e for e in crai).encode(), mtime=0))


def _mate_plan(rs: List[dict]) -> List[Tuple[str, int]]:
    """How each record of a slice stores its mate: ("attached", NF) and ("last", 0) for a pair whose in-slice fix-up
    (cram.cu) reproduces next ref, next pos, TLEN and flags exactly; ("none", 0) for a record whose mate fields are
    empty and that is not paired; ("detached", 0) otherwise."""
    plan = [("detached", 0)] * len(rs)
    for j, r in enumerate(rs):
        if not r["flag"] & 0x1 and r["nrid"] == -1 and r["npos"] == -1 and r["tlen"] == 0 and not r["flag"] & 0x28:
            plan[j] = ("none", 0)
    by_name: Dict[bytes, List[int]] = {}
    for j, r in enumerate(rs):
        if r["flag"] & 0x1 and not r["flag"] & 0x900:
            by_name.setdefault(r["name"], []).append(j)
    for name, js in by_name.items():
        if len(js) != 2:
            continue
        a, b = js
        if _fixup_matches(rs[a], rs[b]):
            plan[a] = ("attached", b - a - 1)
            plan[b] = ("last", 0)
    return plan


def _fixup_matches(ra: dict, rb: dict) -> bool:
    """Whether the decoder's fix-up of an attached pair gives both records their stored mate fields and flags."""
    def apos(r):
        return r["pos"] + 1

    def aend(r):
        if r["flag"] & 0x4:
            return apos(r)
        return apos(r) + max(_ref_len(r["cigar"]), 1) - 1
    aleft = min(apos(ra), apos(rb))
    left_cnt = (apos(ra) == aleft) + (apos(rb) == aleft)
    aright = max(aend(ra), aend(rb))
    same = ra["rid"] == rb["rid"]
    tl = aright - aleft + 1
    for r, m in ((ra, rb), (rb, ra)):
        if not same:
            t = 0
        elif apos(r) == aleft and (left_cnt == 1 or r["flag"] & 0x40):
            t = tl
        else:
            t = -tl
        fl = (r["flag"] & ~0x28) | 0x1
        if m["flag"] & 0x4:
            fl |= 0x8
            t = 0
        if fl & 0x4:
            t = 0
        if m["flag"] & 0x10:
            fl |= 0x20
        if (fl, t, m["rid"], m["pos"]) != (r["flag"], r["tlen"], r["nrid"], r["npos"]):
            return False
    return True
