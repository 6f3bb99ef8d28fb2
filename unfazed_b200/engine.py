"""Batch engine: columnar tables + a window plan -> device pipeline -> per-DNM results.

PyTorch is used only for device memory, streams and events; every kernel is in
``libunfazed_sm100.so`` and is reached through the C ABI (``_lib.py``).  There is no CPU fallback:
constructing an ``Engine`` without the library or without a GPU raises.

Pipeline (one stream, in order):

  K0 window_search -> scan -> K1 classify_sites -> compact_sites -> scan(row marks)
  -> K2 read_scan -> scan(hit counts) -> K3 read_site_alleles
  -> chain_size -> 6 scans -> K4 chain_tally -> K5 summarize
"""
from __future__ import annotations

import contextlib
import ctypes as C
import collections
import os
import time
from dataclasses import dataclass, field
from typing import Dict, List, Optional

import numpy as np
import torch

from . import _lib as L
from .plan import Plan
from .schema import ReadTable, SiteTable, min_base_qual


def make_params(ab_homref=(0.0, 0.2), ab_homalt=(0.8, 1.0), ab_het=(0.2, 0.8), min_gt_qual=20, min_depth=10,
                min_map_qual=1, readlen=151, insert_size_max_sample=1000000, no_extended=False,
                evidence_min_ratio=10, split_error_margin=5) -> L.Params:
    p = L.Params()
    p.ab_homref[0], p.ab_homref[1] = float(ab_homref[0]), float(ab_homref[1])
    p.ab_homalt[0], p.ab_homalt[1] = float(ab_homalt[0]), float(ab_homalt[1])
    p.ab_het[0], p.ab_het[1] = float(ab_het[0]), float(ab_het[1])
    p.min_gt_qual = float(min_gt_qual)
    p.min_depth = int(min_depth)
    p.min_map_qual = int(min_map_qual)
    p.readlen = int(readlen)
    p.ext_read_goal = int(min(insert_size_max_sample, 2**31 - 1))
    p.no_extended = int(bool(no_extended))
    p.evidence_min_ratio = int(evidence_min_ratio)
    p.split_error_margin = int(split_error_margin)
    return p


def pack_site_rows(pos, flag, gt, gq, rd, ad):
    """Device-side repack of the SoA genotype columns into the classifier's row layout
    (meta u32, rec 4xf32, dep 6xi32 -- see include/unfazed_sm100.h).  All torch ops on the device."""
    g = gt.to(torch.int32)
    meta = (flag.to(torch.int32) | (g[0] << 8) | (g[1] << 16) | (g[2] << 24)).contiguous()
    rec = torch.stack([pos.view(torch.float32), gq[0], gq[1], gq[2]], dim=1).contiguous()
    dep = torch.stack([rd[0], ad[0], rd[1], ad[1], rd[2], ad[2]], dim=1).contiguous()
    return meta, rec, dep


class DeviceSites:
    def __init__(self, table: SiteTable, device: torch.device, pin: bool = False, engine: "Engine" = None):
        self.table = table
        self.n_rows = table.n_rows
        up = lambda a: _to_device(np.ascontiguousarray(a), device, pin)
        self.blk_off = up(table.blk_off.astype(np.int64))
        self.pos, self.ref, self.alt = up(table.pos), up(table.ref), up(table.alt)
        flag, gt, gq, rd, ad = up(table.flag), up(table.gt), up(table.gq), up(table.rd), up(table.ad)
        self.h2d_bytes = sum(t.numel() * t.element_size() for t in (self.pos, self.ref, self.alt, flag, gt, gq, rd, ad))
        if engine is not None:
            V = max(self.n_rows, 1)
            self.meta = torch.empty((V,), dtype=torch.int32, device=device)
            self.rec = torch.empty((V, 4), dtype=torch.float32, device=device)
            self.dep = torch.empty((V, 6), dtype=torch.int32, device=device)
            st = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
            engine._check(engine.lib.unfz_pack_site_rows(engine.ctx, self.n_rows, self.pos.data_ptr(), flag.data_ptr(), gt.data_ptr(),
                                                         gq.data_ptr(), rd.data_ptr(), ad.data_ptr(), self.meta.data_ptr(),
                                                         self.rec.data_ptr(), self.dep.data_ptr(), st), "pack_site_rows")
        else:
            self.meta, self.rec, self.dep = pack_site_rows(self.pos, flag, gt, gq, rd, ad)
        self.cols = make_site_cols(table.n_rows, table.n_blocks, self.blk_off, self.pos, self.ref, self.alt,
                                   self.meta, self.rec, self.dep)

    @property
    def nbytes(self) -> int:
        return self.h2d_bytes


def make_site_cols(n_rows, n_blocks, blk_off, pos, ref, alt, meta, rec, dep) -> L.SiteCols:
    c = L.SiteCols()
    c.n_rows, c.n_blocks = n_rows, n_blocks
    c.blk_off, c.pos, c.ref, c.alt = blk_off.data_ptr(), pos.data_ptr(), ref.data_ptr(), alt.data_ptr()
    c.meta, c.rec, c.dep = meta.data_ptr(), rec.data_ptr(), dep.data_ptr()
    return c


class PackedReads:
    """The read columns exactly as they cross PCIe (optionally in pinned memory): 32-byte headers,
    CIGAR words, the low-quality bit plane for ONE base-quality threshold, 2-bit bases and the sorted
    index list of the non-ACGT bases.  A packer that decodes a BAM can fill this directly; tables that
    carry quality bytes (synthetic data, the oracle's fixtures) are reduced here."""

    def __init__(self, table: ReadTable, min_bq: int, pin: bool = False):
        if table.qual is None:
            raise ValueError("PackedReads needs the quality bytes and bases of the table; this ReadTable was decoded on "
                             "the device (bamio.read_regions(engine=...)): use its device_reads")
        self.table, self.min_bq = table, int(min_bq)
        conv = (lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()) if pin else np.ascontiguousarray
        self.hdr = conv(table.hdr.view(np.uint8).reshape(-1))
        self.cigar = conv(table.cigar)
        self.lowq = conv(table.lowq_plane(self.min_bq))
        self.seq2 = conv(table.seq2)
        self.nidx = conv(table.n_index())

    @property
    def nbytes(self) -> int:
        return sum(int(a.nbytes) for a in (self.hdr, self.cigar, self.lowq, self.seq2, self.nidx))


class DeviceReads:
    def __init__(self, table, device: torch.device, pin: bool = False, min_bq: int = 20, engine: "Engine" = None):
        packed = table if isinstance(table, PackedReads) else PackedReads(table, min_bq)
        table = packed.table
        self.table, self.min_bq = table, packed.min_bq
        self.n_reads = table.n_reads
        self.max_l_seq = table.max_l_seq()
        up = lambda a, pad=0: _to_device(a, device, pin, pad)
        self.blk_off = up(np.ascontiguousarray(table.blk_off.astype(np.int64)))
        self.hdr = up(packed.hdr)
        self.cigar = up(packed.cigar)
        # tail padding: the scan's asynchronous copies round the staged span up to 16 B; planes are read as words
        nq = int(table.qual.shape[0])
        plane_bytes = (nq + 7) // 8
        self.lowq = up(packed.lowq, 48 + (-plane_bytes) % 4)
        self.seq2 = up(packed.seq2, 16)
        self.nidx = up(packed.nidx)
        self.nmask = torch.zeros(self.lowq.shape[0], dtype=torch.uint8, device=device)
        self.h2d_bytes = packed.nbytes
        st = self._bind_cols(table, device, nq)
        if engine is not None:
            engine._check(engine.lib.unfz_read_starts(engine.ctx, C.byref(self.cols), self.start.data_ptr(), st), "read_starts")
        else:
            self.start.copy_(self.hdr.view(torch.int32).view(-1, 8)[:, 0]) if table.n_reads else None
        if engine is not None and packed.nidx.shape[0]:
            engine._check(engine.lib.unfz_expand_nlist(engine.ctx, C.byref(self.cols), self.hdr.data_ptr(), self.nmask.data_ptr(),
                                                       self.nidx.data_ptr(), int(packed.nidx.shape[0]), st), "expand_nlist")

    @classmethod
    def from_bam(cls, table: ReadTable, device: torch.device, min_bq: int, engine: "Engine", dbuf: torch.Tensor,
                 dsrc: torch.Tensor) -> "DeviceReads":
        """The read columns decoded on the device from inflated BAM records (``dbuf``; ``dsrc[r]``: byte offset of the
        record of read r): the headers of the host table go up, the CIGAR words and the three base planes are written
        by unfz_bam_emit_cigar / unfz_bam_emit_planes, exactly as an upload of the host-decoded table leaves them.
        One difference in the path, not in the result: there is no sparse index list of the non-ACGT bases
        (``nidx`` stays empty, unfz_expand_nlist does not run) -- the planes kernel owns whole 32-base words, so it
        writes the ``nmask`` words and sets aux bit7 of their reads itself; nothing downstream reads ``nidx``."""
        self = cls.__new__(cls)
        self.table, self.min_bq = table, int(min_bq)
        self.n_reads = table.n_reads
        self.max_l_seq = table.max_l_seq()
        up = lambda a: _to_device(a, device, False)
        self.blk_off = up(np.ascontiguousarray(table.blk_off.astype(np.int64)))
        self.hdr = up(table.hdr.view(np.uint8).reshape(-1))
        nq = table.n_qual
        plane_bytes = (nq + 7) // 8
        self.cigar = torch.empty((int(table.cigar.shape[0]),), dtype=torch.int32, device=device)
        self.lowq = torch.zeros((plane_bytes + 48 + (-plane_bytes) % 4,), dtype=torch.uint8, device=device)
        self.seq2 = torch.zeros(((nq + 3) // 4 + 16,), dtype=torch.uint8, device=device)
        self.nidx = torch.zeros((0,), dtype=torch.int64, device=device)
        self.nmask = torch.zeros(self.lowq.shape[0], dtype=torch.uint8, device=device)
        self.h2d_bytes = int(table.hdr.nbytes + table.blk_off.nbytes)
        st = self._bind_cols(table, device, nq)
        lib, ctx, c = engine.lib, engine.ctx, C.byref(self.cols)
        engine._check(lib.unfz_bam_emit_cigar(ctx, c, dbuf.data_ptr(), dsrc.data_ptr(), st), "bam_emit_cigar")
        engine._check(lib.unfz_read_starts(ctx, c, self.start.data_ptr(), st), "read_starts")
        engine._check(lib.unfz_bam_emit_planes(ctx, c, dbuf.data_ptr(), dsrc.data_ptr(), int(min_bq), st), "bam_emit_planes")
        return self

    def _bind_cols(self, table, device, nq):
        self.blk_sblk = torch.full((max(table.n_blocks, 1),), -1, dtype=torch.int32, device=device)
        self.blk_cul = torch.zeros((max(table.n_blocks, 1),), dtype=torch.float64, device=device)
        c = L.ReadCols()
        c.n_reads, c.n_blocks = table.n_reads, table.n_blocks
        c.blk_off, c.blk_sblk, c.blk_cul = self.blk_off.data_ptr(), self.blk_sblk.data_ptr(), self.blk_cul.data_ptr()
        self.start = torch.empty((max(table.n_reads, 1),), dtype=torch.int32, device=device)
        c.hdr, c.cigar, c.seq2 = self.hdr.data_ptr(), self.cigar.data_ptr(), self.seq2.data_ptr()
        c.start = self.start.data_ptr()
        c.lowq, c.nmask = self.lowq.data_ptr(), self.nmask.data_ptr()
        c.n_qual, c.n_cigar = nq, int(table.cigar.shape[0])
        self.cols = c
        return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)

    @property
    def nbytes(self) -> int:
        """Bytes that crossed PCIe for these columns."""
        return self.h2d_bytes


class _Decoder:
    """What the device decoders share: the bytes that crossed PCIe each way, the device time of every stage by name
    (``timings_ms``, accumulated over calls), and the upload, launch and two-pass output they all use."""

    def __init__(self, engine: "Engine"):
        self.engine = engine
        self.h2d_bytes = self.d2h_bytes = 0
        self.timings_ms: Dict[str, float] = {}

    @contextlib.contextmanager
    def _stages(self):
        """Context on the engine's stream that yields ``mark``: ``mark(name)`` records an event that closes the
        interval ``name``, begun at the previous mark (or on entry); ``mark(None)`` begins an interval without timing
        the gap before it.  On a normal exit every interval is added to ``timings_ms``, read once the last event has
        completed."""
        marks = []

        def mark(name):
            ev = torch.cuda.Event(enable_timing=True)
            ev.record(self.engine.stream)
            marks.append((name, ev))
        with self.engine.on_stream():
            mark(None)
            yield mark
        marks[-1][1].synchronize()
        for (_, e0), (name, e1) in zip(marks, marks[1:]):
            if name is not None:
                self.timings_ms[name] = self.timings_ms.get(name, 0.0) + e0.elapsed_time(e1)

    def _up(self, a: np.ndarray, dtype=None, pad: int = 0, fill: int = 0) -> torch.Tensor:
        """Host array -> device through pinned staging (+ ``pad`` zero elements), its bytes counted in ``h2d_bytes``.
        An empty array becomes one 16-byte buffer with ``fill`` in every element, so a kernel that is told there are no
        items still gets a valid address (``fill=-1`` for a ``slot_of``: no column)."""
        a = np.ascontiguousarray(a, dtype=dtype)
        self.h2d_bytes += int(a.nbytes)
        if a.shape[0]:
            return _to_device(a, self.engine.device, True, pad)
        t = torch.from_numpy(a.view(np.uint8) if a.dtype.fields is not None else a)
        return torch.full((16 // t.element_size(),), fill, dtype=t.dtype, device=self.engine.device)

    def _launch(self, fn: str, *args) -> None:
        """``lib.<fn>(ctx, *args, stream)`` on the engine's stream, a tensor passed by its device address; raises
        with the library's message when it fails."""
        eng = self.engine
        args = [a.data_ptr() if isinstance(a, torch.Tensor) else a for a in args]
        eng._check(getattr(eng.lib, fn)(eng.ctx, *args, C.c_void_p(eng.stream.cuda_stream)), fn)

    def _scan(self, lens: torch.Tensor, off: torch.Tensor, n: int) -> None:
        """``off[0..n]``: the exclusive scan of ``lens[:n]``, ``off[n]`` the total."""
        self._launch("unfz_exclusive_scan_i64", lens, off, n, self.engine._scan_work(n))

    def _size_scan(self, mark, names, n: int, n_status: int, status_dtype, size):
        """First pass of an output of ``n`` items of variable length: ``size(out_len, status)`` launches the kernel
        that writes the length of every item to ``out_len[:n]`` and the statuses (``n_status`` zeroed elements of
        ``status_dtype``); ``_scan`` places the items; the statuses and the total come down in one copy, for the
        caller to check before ``_write``.  ``names``: the timed intervals (``mark``) that end after the size kernel,
        the scan and the download.  Returns (out_len, offsets, device status, host status, total)."""
        eng = self.engine
        out_len = eng._empty(n, torch.int64)
        off = torch.empty((n + 1,), dtype=torch.int64, device=eng.device)
        # the statuses, then the total at the next multiple of 8 bytes: one download
        sb = n_status * torch.iinfo(status_dtype).bits // 8
        nb = (sb + 7) // 8 * 8
        stat = torch.zeros((nb + 8,), dtype=torch.uint8, device=eng.device)
        status = stat[:sb].view(status_dtype)
        size(out_len, status)
        mark(names[0])
        self._scan(out_len, off, n)
        mark(names[1])
        stat[nb:].view(torch.int64).copy_(off[n:])
        host = stat.cpu()
        mark(names[2])
        self.d2h_bytes += nb + 8
        return out_len, off, status, host[:sb].view(status_dtype).numpy(), int(host[nb:].view(torch.int64)[0])

    def _write(self, mark, names, total: int, write, out: Optional[torch.Tensor] = None) -> np.ndarray:
        """Second pass: ``write(out)`` launches the kernel that writes the items into ``out`` (``total`` bytes unless
        the caller passes one), and the output comes down in one copy.  ``names``: the timed intervals (``mark``)
        that end after the kernel and after the download; the gap before the kernel is not timed."""
        if out is None:
            out = self.engine._empty(total, torch.uint8)
        mark(None)
        write(out)
        mark(names[0])
        # one copy into pageable memory (the driver stages it): page-locking a fresh block of the output's size costs
        # more than the copy itself
        host = out[:total].cpu()
        mark(names[1])
        self.d2h_bytes += total
        return host.numpy()


class BamDecoder(_Decoder):
    """Device side of ``bamio.read_regions(engine=...)``: the inflated record bytes go up once (pinned), the fixed
    fields are parsed there (unfz_bam_parse) and come back for the host's selection, and the bulk columns are emitted
    on the device.  The record bytes stay resident, so the planes of another base-quality threshold are decoded again
    from them (``device_reads``) without touching the file.  Resident means every record of the fetched chunks, not
    only the selected reads (1.5 GB with offsets for the 4.4 M reads of 2000 c2 DNMs, profiles/r3_bam_decode_c2_2000dnms.json);
    with several files the parts are concatenated once on the device, which briefly holds both copies."""

    def __init__(self, engine: "Engine"):
        super().__init__(engine)
        self.parts: List[torch.Tensor] = []
        self.dbuf = self.dsrc = self.table = None
        self._reads: Optional[DeviceReads] = None

    def parse(self, buf: np.ndarray, offs: np.ndarray, part: int) -> np.ndarray:
        n = int(offs.shape[0])
        rsz = L.BAM_REC_DTYPE.itemsize
        with self._stages() as mark:
            d = buf.resident if isinstance(buf, ResidentBytes) else None   # records decoded on this GPU stay there
            if d is None:
                d = self._up(buf, pad=16)
            doffs = self._up(offs, np.int64)
            mark("h2d_records")
            out = self.engine._empty(n * rsz, torch.uint8)
            self._launch("unfz_bam_parse", d, int(buf.shape[0]), doffs, n, out)
            mark("parse")
            rec = out[: n * rsz].cpu().numpy().view(L.BAM_REC_DTYPE)
        self.d2h_bytes += int(rec.nbytes)
        bad = int(np.count_nonzero(rec["aux"] & L.BAM_AUX_BAD))
        if bad:
            raise ValueError("%d malformed BAM record(s): fields or aux tags overrun block_size" % bad)
        self.parts.append(d[: int(buf.shape[0])])
        return rec

    def prepare(self, src: np.ndarray) -> None:
        """The parts as one device buffer and the record offset of every output read (``src``: byte offsets in the parts
        back to back)."""
        with self._stages() as mark:
            self.dbuf = torch.cat(self.parts) if len(self.parts) != 1 else self.parts[0]
            if self.dbuf.numel() == 0:
                self.dbuf = torch.zeros((16,), dtype=torch.uint8, device=self.engine.device)
            self.parts = [self.dbuf]
            self.dsrc = self._up(src, np.int64)
            mark("concat_src")

    def mate_join(self, name_hash: np.ndarray, blk: np.ndarray, flag: np.ndarray) -> np.ndarray:
        """Mate index of every output read (after ``prepare``), as packers._mate_join defines it inside each block:
        the reads are ordered by (block, name hash) with torch's stable sort, unfz_bam_mate_join picks the first primary
        read of the other segment in each group and compares the name bytes of every joined pair; -2 marks the reads
        left to the host (a hash collision, or a read that is its own candidate)."""
        n = int(name_hash.shape[0])
        if n == 0:
            return np.zeros(0, dtype=np.int64)
        with self._stages() as mark:
            dh = self._up(np.ascontiguousarray(name_hash).view(np.int64))
            db = self._up(blk, np.int32)
            df = self._up(flag, np.int32)
            o1 = torch.sort(dh, stable=True).indices
            order = o1[torch.sort(db[o1], stable=True).indices].contiguous()
            mate = torch.empty((n,), dtype=torch.int32, device=self.engine.device)
            self._launch("unfz_bam_mate_join", order, dh, db, df, n, self.dbuf, self.dsrc, mate)
            mark("mate_join")
            out = mate.cpu().numpy().astype(np.int64)
        self.d2h_bytes += 4 * n
        return out

    def emit(self, table: ReadTable, min_gt_qual) -> DeviceReads:
        """The DeviceReads of ``table`` (after ``prepare``)."""
        self.table = table
        return self.device_reads(min_gt_qual)

    def device_reads(self, min_gt_qual=20) -> DeviceReads:
        """DeviceReads with the low-quality plane of ``min_gt_qual`` (the last one is kept)."""
        mb = min_base_qual(min_gt_qual)
        if self._reads is None or self._reads.min_bq != mb:
            self._reads = None
            eng = self.engine
            with self._stages() as mark:
                self._reads = DeviceReads.from_bam(self.table, eng.device, mb, eng, self.dbuf, self.dsrc)
                mark("emit")
        return self._reads


class ResidentBytes(np.ndarray):
    """Host bytes with an identical copy on the device (``resident``, 16 bytes of tail padding): ``BamDecoder.parse``
    takes that copy instead of uploading the host one."""
    resident = None


class CramDecoder(_Decoder):
    """Device side of ``cramio.CramFile`` with an engine: the decompressed blocks of the selected slices, their
    descriptors and the reference spans go up; cram_slice_size_kernel sizes every record, unfz_exclusive_scan_i64
    places them, cram_slice_write_kernel writes the BAM records.  The records stay on the device for the BAM stages
    (``ResidentBytes``); a host copy comes back because ``bamio.read_regions`` reads names, CIGARs and the lone mates'
    bytes on the host."""

    def decode(self, cram, desc):
        sl, blocks, ext, prog, ref, rbytes, n_rec, coffs = desc
        eng = self.engine
        n = int(sl.shape[0])
        with self._stages() as mark:
            args = [self._up(np.ascontiguousarray(a).view(np.uint8).reshape(-1), pad=16)
                    for a in (sl, blocks, ext, prog, ref, rbytes)]
            args.insert(1, n)
            mark("h2d")
            rec_cig = eng._zeros(n_rec, torch.int32)
            _, offs, status, stat, total = self._size_scan(
                mark, ("size", "scan", None), n_rec, n, torch.int32,
                lambda rec_len, st: self._launch("unfz_cram_decode_size", *args, rec_len, rec_cig, st))
            cram.check_status(stat, coffs)
            # zeroed: the write step ORs the bases into place, two to a byte, and the 16-byte tail stays zero
            out = torch.zeros((total + 16,), dtype=torch.uint8, device=eng.device)
            host = self._write(mark, ("write", None), total,
                               lambda out: self._launch("unfz_cram_decode_write", *args, rec_cig, offs, out, status), out)
            stat = status.cpu().numpy()
            hoffs = offs[:n_rec].cpu().numpy()
        self.d2h_bytes += int(stat.nbytes + hoffs.nbytes)
        cram.check_status(stat, coffs)
        buf = host.view(ResidentBytes)
        buf.resident = out
        return buf, hoffs


_CELLS = (("gt", torch.uint8), ("gq", torch.float32), ("rd", torch.int32), ("ad", torch.int32), ("status", torch.uint8))


class VcfDecoder(_Decoder):
    """Device side of ``vcfio.read_sites(engine=...)``, with the calls of ``vcfio.HostDecoder``: the inflated text goes
    up once (pinned staging), the newline pass (unfz_vcf_line_count, a scan, unfz_vcf_line_write) and the fixed-field
    parse (unfz_vcf_parse) run on the engine's stream and the 64-byte records come back for the host's selection; then
    unfz_vcf_samples decodes the member columns of the selected lines, which come back as the table's genotype arrays.
    The floats it leaves to the host are decoded by ``vcfio.finish_cells``.  ``rewrite`` writes the phased VCF body from
    the same resident text and records (``vcfio.write_phased_vcf``)."""

    def lines(self, buf: np.ndarray) -> np.ndarray:
        eng = self.engine
        n = int(buf.shape[0])
        chunks = int(eng.lib.unfz_vcf_chunks(n))
        rsz = L.VCF_REC_DTYPE.itemsize
        with self._stages() as mark:
            # 16 bytes of padding: the sample pass reads whole 16-byte words
            self.dbuf = self._up(buf, pad=16)
            mark("h2d_text")
            cnt = eng._empty(chunks, torch.int32)
            at = torch.empty((chunks + 1,), dtype=torch.int32, device=eng.device)
            total = torch.zeros((1,), dtype=torch.int64, device=eng.device)
            self._launch("unfz_vcf_line_count", self.dbuf, n, cnt)
            self._launch("unfz_exclusive_scan_u32", cnt, at, chunks, total, eng._scan_work(chunks))
            n_lines = self.n_lines = int(total.item())
            self.ends = eng._empty(n_lines, torch.int64)
            self._launch("unfz_vcf_line_write", self.dbuf, n, at, self.ends)
            mark("line_bounds")
            self.drecs = eng._empty(n_lines * rsz, torch.uint8)
            self._launch("unfz_vcf_parse", self.dbuf, self.ends, n_lines, self.drecs)
            mark("parse")
            recs = self.drecs[: n_lines * rsz].cpu().numpy().view(L.VCF_REC_DTYPE)
            mark("d2h_records")
        self.d2h_bytes += int(recs.nbytes) + 8
        return recs

    def samples(self, sel: np.ndarray, slot_of: np.ndarray, n_members: int, gq_float: bool,
                max_digits: int = 15) -> Dict[str, np.ndarray]:
        eng = self.engine
        ns, m = int(sel.shape[0]), int(n_members)
        cells = ns * m
        with self._stages() as mark:
            dsel = self._up(sel, np.int64)
            dslot = self._up(slot_of, np.int32, fill=-1)
            mark("h2d_select")
            out = {k: eng._empty(cells, dt) for k, dt in _CELLS}
            out["line_bad"] = eng._empty(ns, torch.uint8)
            self._launch("unfz_vcf_samples", self.dbuf, self.drecs, dsel, ns, dslot, int(slot_of.shape[0]), m,
                         int(bool(gq_float)), int(max_digits), *(out[k] for k, _ in _CELLS), out["line_bad"])
            mark("samples")
            host = {k: v.cpu().numpy() for k, v in out.items()}
            mark("d2h_cells")
        self.d2h_bytes += cells * 14 + ns
        res = {k: host[k][:cells].reshape(ns, m) for k, _ in _CELLS}
        res["line_bad"] = host["line_bad"][:ns]
        return res

    def rewrite(self, edit_off: np.ndarray, edits: np.ndarray, n_samples: int):
        """Every line of the text ``lines()`` left on the device, rewritten with the edit list (csrc/vcfout.cu):
        (the output bytes, the status of every line, UNFZ_VCFOUT_*).  Only the edits go up; the line lengths are sized
        (unfz_vcf_rewrite_size), scanned (unfz_exclusive_scan_i64) and written (unfz_vcf_rewrite_write) on the engine's
        stream, and the output comes down in one copy.  With a bad line nothing is written: the output
        is empty and the status says why."""
        n = self.n_lines
        with self._stages() as mark:
            doff = self._up(edit_off, np.int64)
            ded = self._up(edits, L.VCF_EDIT_DTYPE)
            mark("h2d_edits")
            args = (self.dbuf, self.drecs, n, doff, ded, int(n_samples))
            _, off, _, line_bad, total = self._size_scan(
                mark, ("rewrite_size",) * 3, n, n, torch.uint8,
                lambda out_len, stat: self._launch("unfz_vcf_rewrite_size", *args, out_len, stat))
            if line_bad.any():
                return np.zeros(0, dtype=np.uint8), line_bad
            out = self._write(mark, ("rewrite_write", "d2h_output"), total,
                              lambda out: self._launch("unfz_vcf_rewrite_write", *args, off, out))
        return out, line_bad


class BcfDecoder(_Decoder):
    """Device side of ``bcfio.read_sites(engine=...)``, with the calls of ``bcfio.HostDecoder``: the inflated record
    bytes go up once (pinned staging) with the record offsets the host walked, unfz_bcf_parse runs on the engine's stream
    and the 80-byte records come back for the host's selection; then unfz_bcf_samples decodes the member cells of the
    selected records -- one thread per cell, a direct load at the field's sample stride -- which come back as the
    table's genotype arrays."""

    def records(self, buf: np.ndarray, offs: np.ndarray, keys: np.ndarray, n_samples: int) -> np.ndarray:
        n = int(offs.shape[0])
        rsz = L.BCF_REC_DTYPE.itemsize
        keys = np.ascontiguousarray(keys, dtype=np.int32)
        with self._stages() as mark:
            self.buf = buf
            self.dbuf = self._up(buf)
            doffs = self._up(offs, np.int64)
            mark("h2d_records")
            self.drecs = self.engine._empty(n * rsz, torch.uint8)
            self._launch("unfz_bcf_parse", self.dbuf, doffs, n, keys.ctypes.data, int(n_samples), self.drecs)
            mark("parse")
            recs = self.drecs[: n * rsz].cpu().numpy().view(L.BCF_REC_DTYPE)
            mark("d2h_records")
        self.d2h_bytes += int(recs.nbytes)
        self.recs = recs
        return recs

    def samples(self, sel: np.ndarray, member_sample: np.ndarray) -> Dict[str, np.ndarray]:
        ns, m = int(sel.shape[0]), int(member_sample.shape[0])
        cells = ns * m
        with self._stages() as mark:
            dsel = self._up(sel, np.int64)
            dms = self._up(member_sample, np.int32)
            mark("h2d_select")
            out = {k: self.engine._empty(cells, dt) for k, dt in _CELLS}
            self._launch("unfz_bcf_samples", self.dbuf, self.drecs, dsel, ns, dms, m, *(out[k] for k, _ in _CELLS))
            mark("samples")
            host = {k: v.cpu().numpy() for k, v in out.items()}
            mark("d2h_cells")
        self.d2h_bytes += cells * 14
        return {k: host[k][:cells].reshape(ns, m) for k, _ in _CELLS}

    def format(self, edit_off: np.ndarray, edits: np.ndarray, n_samples: int, names, fkeys: np.ndarray):
        """The records ``records()`` left on the device printed as the phased VCF body (csrc/bcfout.cu): (the output
        bytes, the status of every record, UNFZ_BCFOUT_*), as ``bcfio.HostDecoder.format``.  Only the edits and the
        dictionaries go up; the record lengths are sized (unfz_bcf_format_size), scanned (unfz_exclusive_scan_i64) and
        written (unfz_bcf_format_write) on the engine's stream, the statuses and the total come down in one copy and
        the output in another.  A record with a float off the device's exact path is printed by the host entry points
        (``bcfio.format_host``): its length goes up before a second scan, and its text is copied into its slot.  With
        a haploid phase edit or a malformed record nothing is written: the output is empty and the status says why."""
        from .bcfio import format_host
        n = int(self.recs.shape[0])
        fkeys = np.ascontiguousarray(fkeys, dtype=np.int32)
        with self._stages() as mark:
            doff = self._up(edit_off, np.int64)
            ded = self._up(edits, L.VCF_EDIT_DTYPE)
            dnames = [self._up(a) for a in names]
            mark("h2d_edits")
            args = (self.dbuf, self.drecs, n, dnames[0], dnames[1], int(names[1].shape[0]) - 1, dnames[2], dnames[3],
                    int(names[3].shape[0]) - 1, fkeys.ctypes.data, doff, ded, int(n_samples))
            out_len, off, dstat, status, total = self._size_scan(
                mark, ("format_size",) * 3, n, n, torch.uint8,
                lambda out_len, stat: self._launch("unfz_bcf_format_size", *args, out_len, stat))
            if (status & (L.BCFOUT_HAPLOID | L.BCFOUT_BAD)).any():
                return np.zeros(0, dtype=np.uint8), status
            host = np.flatnonzero(status & L.BCFOUT_FLOAT_HOST)
            if host.shape[0]:
                # the host prints these records; their lengths replace the device's before the offsets are scanned again
                t0 = time.perf_counter()
                cnt = edit_off[host + 1] - edit_off[host]
                sub_off = np.zeros(host.shape[0] + 1, dtype=np.int64)
                np.cumsum(cnt, out=sub_off[1:])
                sub_edits = edits[np.repeat(edit_off[host] - sub_off[:-1], cnt) + np.arange(int(sub_off[-1]))]
                text, _st, lens = format_host(self.buf, self.recs[host], sub_off, sub_edits, n_samples, names, fkeys)
                self.timings_ms["format_host"] = self.timings_ms.get("format_host", 0.0) + 1e3 * (time.perf_counter() - t0)
                didx = self._up(host, np.int64)
                out_len[didx] = self._up(lens)
                self._scan(out_len, off, n)
                total = int(off[n:].cpu()[0])
                slot = off[didx].cpu().numpy()
                self.d2h_bytes += 8 + 8 * int(host.shape[0])
            res = self._write(mark, ("format_write", "d2h_output"), total,
                              lambda out: self._launch("unfz_bcf_format_write", *args, dstat, off, out))
        if host.shape[0]:
            src = np.zeros(host.shape[0] + 1, dtype=np.int64)
            np.cumsum(lens, out=src[1:])
            for k in range(host.shape[0]):
                res[int(slot[k]): int(slot[k]) + int(lens[k])] = text[int(src[k]): int(src[k + 1])]
        return res, status


def _to_device(a: np.ndarray, device, pin: bool, pad: int = 0) -> torch.Tensor:
    """Host array -> device tensor (+ ``pad`` zero elements).  Arrays that already live in pinned
    memory are copied asynchronously; ``pin`` stages pageable arrays through a pinned copy."""
    t = torch.from_numpy(a.view(np.uint8).reshape(-1)) if a.dtype.fields is not None else torch.from_numpy(a)
    # small pageable arrays are staged through pinned memory too: a pageable source makes the host wait for the stream
    if not t.is_pinned() and (pin or t.numel() * t.element_size() <= (1 << 20)):
        t = t.pin_memory()
    out = torch.empty(t.shape[:-1] + (t.shape[-1] + pad,), dtype=t.dtype, device=device) if pad else torch.empty_like(t, device=device)
    if pad:
        out[..., t.shape[-1]:].zero_()
        out[..., : t.shape[-1]].copy_(t, non_blocking=True)
    else:
        out.copy_(t, non_blocking=True)
    return out


@dataclass
class BatchResult:
    plan: Plan
    n_pairs: int
    n_hits: int
    seg_row_lo: np.ndarray
    seg_pair_off: np.ndarray
    n_het: np.ndarray
    n_cand: np.ndarray
    cnv_dad: np.ndarray
    cnv_mom: np.ndarray
    tally: Optional[np.ndarray] = None
    calls_strict: Optional[np.ndarray] = None
    calls_ambiguous: Optional[np.ndarray] = None
    win: Optional[np.ndarray] = None          # [4, n]: read-index ranges [a_lo,a_hi) U [b_lo,b_hi) of every entry
    slot_off: Optional[np.ndarray] = None
    # evidence lists (Engine.run(evidence=True)): off int64[4][n+1] (dad pairs, mom pairs, dad sites, mom sites) and the
    # four int32 lists read_dad / read_mom (read indices) / pos_dad / pos_mom (site positions)
    ev: Optional[dict] = None
    timings_ms: Dict[str, float] = field(default_factory=dict)
    launches: int = 0
    _dev: dict = field(default_factory=dict)

    # lazily downloaded bulk outputs ------------------------------------------------------
    def _np(self, name):
        key = "_np_" + name
        if key not in self._dev:
            self._dev[key] = self._dev[name].cpu().numpy()
        return self._dev[key]

    def class_codes(self) -> np.ndarray:
        return self._np("cls")

    def het_rows(self, d: int) -> np.ndarray:
        base = int(self.seg_pair_off[self.plan.dnm["seg_lo"][d]]) if self.plan.dnm["seg_hi"][d] > self.plan.dnm["seg_lo"][d] else 0
        return self._np("het_list")[base: base + int(self.n_het[d])]

    def cand_words(self, d: int) -> np.ndarray:
        base = int(self.seg_pair_off[self.plan.dnm["seg_lo"][d]]) if self.plan.dnm["seg_hi"][d] > self.plan.dnm["seg_lo"][d] else 0
        return self._np("cand_list")[base: base + int(self.n_cand[d])]

    def cand_evidence(self, d: int) -> np.ndarray:
        base = int(self.seg_pair_off[self.plan.dnm["seg_lo"][d]]) if self.plan.dnm["seg_hi"][d] > self.plan.dnm["seg_lo"][d] else 0
        return self._np("cand_evid")[base: base + int(self.n_cand[d])]

    def slot_labels(self, d: int) -> np.ndarray:
        a, b = int(self.slot_off[d]), int(self.slot_off[d + 1])
        return self._np("slot_label")[a:b]

    def slot_evidence(self, d: int) -> np.ndarray:
        a, b = int(self.slot_off[d]), int(self.slot_off[d + 1])
        return self._np("slot_evid")[a:b]

    def slot_reads(self, d: int, slots: np.ndarray) -> np.ndarray:
        """Read index behind window slots of entry d."""
        a_lo, a_hi, b_lo, _b_hi = (int(x) for x in self.win[:, d])
        na = a_hi - a_lo
        slots = np.asarray(slots, dtype=np.int64)
        return np.where(slots < na, a_lo + slots, b_lo + (slots - na))

    def read_summaries(self) -> np.ndarray:
        return self._np("rsum").view(L.RSUM_DTYPE)


class PendingBatch:
    """A batch whose launches are on the stream but whose results have not been waited for
    (``Engine.run(defer=True)``): ``finish()`` waits for THIS batch's download only, so the next batch's copies and
    kernels, already queued behind it, keep the GPU busy while the host turns these results into records."""

    def __init__(self, finish):
        self._finish = finish

    def finish(self) -> "BatchResult":
        f, self._finish = self._finish, None
        if f is None:
            raise RuntimeError("PendingBatch.finish() called twice")
        return f()


class Engine:
    """One engine per (process, GPU)."""

    def __init__(self, device: int = 0):
        if not torch.cuda.is_available():
            raise RuntimeError("unfazed_b200 needs a CUDA device (sm_100a); none is visible -- there is no CPU path")
        self.lib = L.load()
        self.device = torch.device("cuda", device)
        torch.cuda.set_device(self.device)
        ctx = C.c_void_p()
        rc = self.lib.unfz_ctx_create(device, C.byref(ctx))
        if rc != 0:
            raise RuntimeError("unfz_ctx_create failed (%d): libunfazed_sm100.so targets sm_100a only" % rc)
        self.ctx = ctx
        # everything the engine does runs on its own stream: CUDA cannot capture the legacy default stream, and the
        # batch is replayed as a CUDA graph (unfz_run_batch_graph)
        self.stream = torch.cuda.Stream(self.device)
        self.stream2 = torch.cuda.Stream(self.device)      # late downloads of a deferred batch (see PendingBatch)
        self.use_graph = not os.environ.get("UNFZ_NO_GRAPH")
        self._caps = None                                  # capacities seen so far (speculative sizing)
        self.spec_fallbacks = 0                            # batches re-run with exact sizes because a capacity was exceeded
        self._pinned_free: Dict[int, list] = {}            # recycled pinned download blocks by size class
        self._stage_new: list = []                         # pinned upload staging blocks handed out, no event yet
        self._stage_busy: list = []                        # (block, event recorded after its copy)
        self._pool_limit = int(0.35 * torch.cuda.get_device_properties(self.device).total_memory)   # recycled arena bytes

    def on_stream(self):
        """Context: torch's current stream is the engine's (uploads, runs, events recorded by callers)."""
        cur = torch.cuda.current_stream(self.device)
        if cur == self.stream:
            return contextlib.nullcontext()
        self.stream.wait_stream(cur)
        return torch.cuda.stream(self.stream)

    def __del__(self):
        try:
            if getattr(self, "ctx", None):
                self.lib.unfz_ctx_destroy(self.ctx)
                self.ctx = None
        except Exception:
            pass

    # ------------------------------------------------------------------------------------
    def concordant_upper_lens(self, dreads: "DeviceReads", readlen: int, insert_size_max_sample: int, stdevs: int) -> np.ndarray:
        """Per read block: the reference's estimate_concordant_insert_len of the block's kid
        (read_collector.py:11-25), with the order statistics selected on the GPU
        (unfz_insert_size_order_stats) and numpy's own interpolation applied to them."""
        with self.on_stream():
            return self._concordant_upper_lens(dreads, readlen, insert_size_max_sample, stdevs)

    def _concordant_upper_lens(self, dreads, readlen, insert_size_max_sample, stdevs):
        t = dreads.table
        lib, dev = self.lib, self.device
        st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        out = np.zeros(max(t.n_blocks, 1), dtype=np.float64)
        nwork = int(lib.unfz_insert_size_work_bytes())
        head = getattr(t, "head_tlen", None) or {}
        for k, kid in enumerate(t.kids):
            blocks = [b for b in range(t.n_blocks) if int(t.blk_kid[b]) == k]
            cols = dreads.cols
            if kid in head:
                # packed from a real file: the estimate is made over the HEAD of the BAM (read_collector.py:11-25), whose
                # template lengths the packer kept on the host.  They go through the same device selection as a
                # one-column stand-in of the header array (only tlen is read).
                h = np.asarray(head[kid][: insert_size_max_sample + 1], dtype=np.int64)
                tmp_hdr = torch.zeros((max(h.shape[0], 1), 8), dtype=torch.int32, device=dev)
                if h.shape[0]:
                    tmp_hdr[: h.shape[0], 1] = torch.from_numpy(h.astype(np.int32)).to(dev)
                cols = L.ReadCols()
                cols.n_reads, cols.n_blocks, cols.hdr = int(h.shape[0]), 0, tmp_hdr.data_ptr()
                first, count = [0], [int(h.shape[0])]
            else:
                first, count, left = [], [], insert_size_max_sample + 1
                for b in blocks:
                    if left <= 0:
                        break
                    lo, hi = int(t.blk_off[b]), int(t.blk_off[b + 1])
                    take = min(left, hi - lo)
                    first.append(lo)
                    count.append(take)
                    left -= take
            n = int(sum(count))
            if n == 0:
                continue
            # neighbourhood of numpy's virtual index (n-1)*0.995 (linear method)
            k0 = int(np.floor((n - 1) * 0.995))
            ranks = np.clip(np.array([k0 - 1, k0, k0 + 1, k0 + 2], dtype=np.int64), 0, n - 1).astype(np.uint64)
            work = torch.zeros(nwork, dtype=torch.uint8, device=dev)
            vals = torch.zeros(4, dtype=torch.int32, device=dev)
            hf, hc = np.array(first, dtype=np.int64), np.array(count, dtype=np.int64)
            self._check(lib.unfz_insert_size_order_stats(self.ctx, C.byref(cols), hf.ctypes.data, hc.ctypes.data, len(first),
                                                         int(readlen), ranks.ctypes.data, work.data_ptr(), vals.data_ptr(), st),
                        "insert_size_order_stats")
            v = vals.cpu().numpy().view(np.uint32).astype(np.int64)
            # an array with the same order statistics around the virtual index; numpy does the rest
            surrogate = np.empty(n, dtype=np.int64)
            r = ranks.astype(np.int64)
            surrogate[: r[1]] = v[0]
            surrogate[r[1]] = v[1]
            surrogate[r[2]:] = v[3]
            surrogate[r[2]] = v[2]
            pct = np.percentile(surrogate, 99.5)
            cul = float(int(np.mean(pct)) + (np.std(pct) * stdevs))
            for b in blocks:
                out[b] = cul
        return out

    def upload_sites(self, table: SiteTable, pin: bool = False) -> DeviceSites:
        if table.n_rows >= 2 ** 30:
            # candidate words carry two flags above a 30-bit row index (include/unfazed_sm100.h, unfz_compact_sites)
            raise ValueError("a SiteTable holds %d rows; one upload is limited to 2^30 - 1 (split the cohort)" % table.n_rows)
        with self.on_stream():
            return DeviceSites(table, self.device, pin, self)

    def upload_reads(self, table, pin: bool = False, min_gt_qual=20) -> DeviceReads:
        """Read columns -> device.  ``table`` is a ReadTable (reduced to the low-quality plane of
        ``min_gt_qual`` first) or a PackedReads (copied as it is)."""
        with self.on_stream():
            return DeviceReads(table, self.device, pin, min_base_qual(min_gt_qual), self)

    def bam_decoder(self) -> BamDecoder:
        """A device decoder for one ``bamio.read_regions`` load."""
        return BamDecoder(self)

    def vcf_decoder(self) -> VcfDecoder:
        """A device decoder for one ``vcfio.read_sites`` load."""
        return VcfDecoder(self)

    def bcf_decoder(self) -> BcfDecoder:
        """A device decoder for one ``bcfio.read_sites`` load."""
        return BcfDecoder(self)

    def cram_decoder(self) -> CramDecoder:
        """The device slice decoder of this engine's ``cramio.CramFile`` loads (timings and bytes accumulate)."""
        if getattr(self, "_cram", None) is None:
            self._cram = CramDecoder(self)
        return self._cram

    def decode_bam(self, paths, regions, head_reads: int = 0, min_gt_qual=20) -> DeviceReads:
        """Indexed BAM files -> DeviceReads, the bulk of the records decoded on this GPU (``bamio.read_regions``).
        ``.table`` is the host half: headers, CIGAR, names, block layout, head template lengths; no bases."""
        from . import bamio
        return bamio.read_regions(paths, regions, head_reads=head_reads, engine=self, min_gt_qual=min_gt_qual).device_reads

    def pack_reads(self, table: ReadTable, min_gt_qual=20, pin: bool = True) -> PackedReads:
        return PackedReads(table, min_base_qual(min_gt_qual), pin)

    def _pinned(self, a: np.ndarray) -> torch.Tensor:
        """Small host array -> pinned staging tensor (the caller copies it to the device right away, on the current
        stream).  A copy out of PAGEABLE memory makes the host wait for everything queued on the stream before it (the
        driver stages it in order), which would serialise a deferred batch behind the previous batch's 2 GB of uploads; a
        pinned source keeps the call asynchronous.  The blocks are recycled by size class once an event recorded after
        their copy has completed: allocating pinned memory is a slow, device-synchronising call, so a steady-state batch
        must not make one."""
        a = np.ascontiguousarray(a)
        nb = int(a.nbytes)
        st = torch.cuda.current_stream(self.device)
        if self._stage_new:                     # handed out by earlier calls: their copies are on the stream by now
            ev = torch.cuda.Event()
            ev.record(st)
            self._stage_busy += [(blk, ev) for blk in self._stage_new]
            self._stage_new = []
        size = 4096
        while size < nb:
            size *= 2
        blk = None
        for i, (b_, ev) in enumerate(self._stage_busy):
            if b_.numel() == size and ev.query():
                blk = b_
                del self._stage_busy[i]
                break
        if blk is None:
            blk = torch.empty((size,), dtype=torch.uint8, pin_memory=True)
        host = blk[:nb]
        if nb:
            host.numpy()[:] = a.reshape(-1).view(np.uint8)
        self._stage_new.append(blk)
        return host.view(torch.from_numpy(np.empty(0, dtype=a.dtype)).dtype).reshape(a.shape)

    def _pinned_block(self, nbytes: int) -> torch.Tensor:
        """A pinned uint8 block of at least ``nbytes`` (power-of-two size classes), recycled through ``_pinned_free``."""
        size = 4096
        while size < nbytes:
            size *= 2
        free = self._pinned_free.get(size)
        return free.pop() if free else torch.empty((size,), dtype=torch.uint8, pin_memory=True)

    def _h2d(self, a: np.ndarray) -> torch.Tensor:
        return self._pinned(a).to(self.device, non_blocking=True)

    def _check(self, rc: int, what: str):
        if rc != 0:
            raise RuntimeError("%s failed (%d): %s" % (what, rc, self.lib.unfz_last_error(self.ctx).decode()))

    def _empty(self, n, dtype):
        return torch.empty((max(int(n), 1),), dtype=dtype, device=self.device)

    def _zeros(self, n, dtype):
        return torch.zeros((max(int(n), 1),), dtype=dtype, device=self.device)

    def _scan_work(self, n):
        return self._empty(self.lib.unfz_scan_work_bytes(int(n)), torch.uint8)

    # ------------------------------------------------------------------------------------
    def run(self, *args, **kw) -> BatchResult:
        with self.on_stream():
            return self._run(*args, **kw)

    def _run(self, dsites: DeviceSites, dreads: Optional[DeviceReads], plan: Plan, params: L.Params,
             blk_cul: Optional[np.ndarray] = None, time_stages: bool = False, download: bool = True,
             keep_device: bool = True, speculative: bool = True, evidence: bool = False, defer: bool = False):
        """One batch through the pipeline.  The sizes of the variable outputs (pairs; hits + chain
        scratch) are only known on the device.  The first batch reads them back (two host syncs); later
        batches allocate from the capacities the engine has seen (+25 %), have the device check them
        (unfz_check_caps) and run without any host round trip -- if a capacity is exceeded the guarded
        kernels return at once and the batch is re-run with exact sizes.  All per-DNM results come back
        in ONE D2H copy.  Device memory comes from three arenas (one torch allocation each)."""
        lib, ctx, dev = self.lib, self.ctx, self.device
        st = torch.cuda.current_stream(dev)
        s = C.c_void_p(st.cuda_stream)
        n, S = int(plan.dnm.shape[0]), int(plan.seg.shape[0])
        V = int(dsites.n_rows)
        N = int(dreads.n_reads) if dreads is not None else 0
        ev: List = []
        launches = 0
        caps = getattr(self, "_caps", None)
        spec = bool(speculative and download and caps is not None)
        reuse = not keep_device and not os.environ.get("UNFZ_NO_ARENA_REUSE")
        # recycled buffers at stable addresses + sizes known up front: the batch is one CUDA graph, which also clears
        # the zero-initialised arenas (no torch fill kernels on the stream)
        graph = bool(spec and not time_stages and reuse and self.use_graph)
        pool = self.__dict__.setdefault("_arena_pool", {})
        arenas: List = []

        def mark(name):
            if time_stages:
                e_ = torch.cuda.Event(enable_timing=True)
                e_.record(st)
                ev.append((name, e_))

        class Arena:
            def __init__(self, zero: bool):
                self.items, self.size, self.zero, self.buf = [], 0, zero, None

            def add(self, name, nbytes):
                self.items.append((name, self.size, int(nbytes)))
                self.size += (int(nbytes) + 255) & ~255

            def alloc(self_, clear=True):
                # a run that keeps nothing on the device hands its buffers back (see the end of run());
                # the next run with the same layout reuses them and only clears the zero-initialised ones
                self_.key = (self_.zero, tuple(self_.items))
                # one FIFO per layout: with several deferred batches in flight the buffer sets rotate in a fixed order,
                # so a batch meets the same addresses (and its instantiated CUDA graph) every time it comes round
                q_ = pool.get(self_.key) if reuse else None
                buf = q_.popleft() if q_ else None
                if buf is None:
                    fn = torch.zeros if self_.zero else torch.empty
                    buf = fn((max(self_.size, 256),), dtype=torch.uint8, device=dev)
                elif self_.zero and clear:
                    buf.zero_()
                self_.buf = buf
                arenas.append(self_)
                base = self_.buf.data_ptr()
                self_.ptr = {nm: base + off for nm, off, _ in self_.items}
                self_.view = {nm: self_.buf[off: off + nb] for nm, off, nb in self_.items}

        # ---- plan upload: one H2D ----------------------------------------------------------------
        # (a plan that is run again -- same object, same device -- is already resident)
        cached = getattr(plan, "_resident", None)
        if cached is not None and cached[0] == dev and cached[2] == (plan.dnm.nbytes, plan.seg.nbytes, plan.alleles.nbytes):
            d_plan = cached[1]
        else:
            hp = np.concatenate([plan.dnm.view(np.uint8).reshape(-1), plan.seg.view(np.uint8).reshape(-1), plan.alleles,
                                 np.zeros(16, np.uint8)])
            d_plan = self._h2d(hp)
            try:
                plan._resident = (dev, d_plan, (plan.dnm.nbytes, plan.seg.nbytes, plan.alleles.nbytes))
            except AttributeError:
                pass
        p_dnm = d_plan.data_ptr()
        p_seg = p_dnm + plan.dnm.nbytes
        p_all = p_seg + plan.seg.nbytes
        sc = C.byref(dsites.cols)
        has_reads = dreads is not None and N > 0 and bool((plan.dnm["rblk"] >= 0).any())
        if has_reads and dreads.min_bq != min_base_qual(params.min_gt_qual):
            raise ValueError("the read columns on the device hold the low-quality plane of base quality < %d, the call "
                             "asks for < %d: upload them again with upload_reads(table, min_gt_qual=...)"
                             % (dreads.min_bq, min_base_qual(params.min_gt_qual)))

        # ---- arena 1: everything whose size is known up front -------------------------------------
        z1, e1 = Arena(True), Arena(False)
        # int32 result block, downloaded with one copy at the end
        r_fields = [("n_het", n), ("n_cand", n), ("cnv_dad", n), ("cnv_mom", n), ("tally", 8 * n), ("calls_s", 4 * n),
                    ("calls_a", 4 * n), ("win", 4 * n), ("seg_row_lo", S)]
        r_off, acc = {}, 0
        for nm, cnt in r_fields:
            r_off[nm] = acc
            acc += cnt
        # everything the host reads back sits at the front of the arena: one contiguous download
        z1.add("result", 4 * acc)
        z1.add("guard", 256)                      # int32 flag + int64 actual[8] at +64
        z1.add("seg_pair_off", 8 * (S + 1))
        want_ev = bool(evidence and has_reads and download)
        if want_ev:
            z1.add("ev_off", 8 * 4 * (n + 1))
        dl_end = z1.size
        if has_reads:
            z1.add("off", 8 * (6 * (n + 1) + 1))
            dl_end += 8 * (n + 1)                 # row 0 of `off` (slot offsets); the totals travel in `guard`
        z1.add("row_mark", V)
        z1.add("mark_prefix", 4 * (V + 1))
        e1.add("seg_count", 8 * S)
        e1.add("scan_work", lib.unfz_scan_work_bytes(max(S, V, N, n) + 1))
        if has_reads:
            z1.add("blk_maxspan", 4 * max(dreads.table.n_blocks, 1))
            z1.add("need", 8 * 6 * n)
            if want_ev:
                z1.add("ev_need", 8 * 4 * n)
            e1.add("rsum", 32 * N)
            tile_reads = int(lib.unfz_read_scan_tile_reads(dreads.max_l_seq))
            n_tiles = (N + tile_reads - 1) // tile_reads
            e1.add("tile_tot", 4 * n_tiles)
            e1.add("tile_base", 4 * (n_tiles + 1))
            e1.add("tile_info", 8 * n_tiles)
        z1.alloc(clear=not graph)
        e1.alloc()
        R = z1.ptr["result"]
        rp = {nm: R + 4 * o for nm, o in r_off.items()}

        # ---- arena 2: per-pair outputs; arena 3: hits + chain scratch + labels ------------------------
        def arena2(n_pairs_):
            z, e = Arena(True), Arena(False)
            e.add("cls", n_pairs_)
            e.add("het_list", 4 * n_pairs_)
            e.add("cand_list", 4 * n_pairs_)
            if has_reads:
                e.add("site_lo", 4 * n_pairs_)
                e.add("site_n", 4 * n_pairs_)
                e.add("seed_win", 16 * n)
            z.add("cand_evid", n_pairs_ + 8)
            if want_ev:
                e.add("ev_pos_dad", 4 * n_pairs_ + 16)
                e.add("ev_pos_mom", 4 * n_pairs_ + 16)
            z.alloc(clear=not graph)
            e.alloc()
            return z, e

        def arena3(totals_, n_hits_):
            z, e = Arena(True), Arena(False)
            nb = lib.unfz_chain_scratch_bytes(*(int(x) for x in totals_), n)
            e.add("hits", 4 * max(n_hits_, 1))
            e.add("scratch", nb)
            z.add("slot_label", int(totals_[0]) + 4)
            z.add("slot_evid", int(totals_[0]) + 4)
            if want_ev:
                e.add("ev_read_dad", 4 * int(totals_[0]) + 16)
                e.add("ev_read_mom", 4 * int(totals_[0]) + 16)
            z.alloc(clear=not graph)
            e.alloc()
            return z, e, nb

        if spec:                                   # sizes come from the capacities: allocate before anything runs
            z2, e2 = arena2(int(caps["pairs"]))
            if has_reads:
                z3, e3, nbytes = arena3(caps["chain"], int(caps["hits"]))
        mark("start")

        def bind_blocks():
            # read block -> site block map and the per-block insert bound: uploaded unless the same plan and
            # bounds are already bound to these read columns
            cul_bytes = None if blk_cul is None else np.ascontiguousarray(blk_cul, dtype=np.float64).tobytes()
            token = getattr(plan, "_token", None)
            if token is None:
                token = object()
                try:
                    plan._token = token
                except AttributeError:
                    pass
            bound = (token, cul_bytes)
            if getattr(dreads, "_bound", None) != bound:
                sb = np.full(max(dreads.table.n_blocks, 1), -1, dtype=np.int32)
                if plan.rblk_sblk:
                    keys = np.fromiter(plan.rblk_sblk.keys(), dtype=np.int64, count=len(plan.rblk_sblk))
                    sb[keys] = np.fromiter(plan.rblk_sblk.values(), dtype=np.int32, count=len(plan.rblk_sblk))
                dreads.blk_sblk.copy_(self._pinned(sb), non_blocking=True)
                if blk_cul is not None:
                    dreads.blk_cul[: blk_cul.shape[0]].copy_(self._pinned(np.frombuffer(cul_bytes, dtype=np.float64).copy()), non_blocking=True)
                dreads._bound = bound

        fast = spec and not time_stages
        if fast:
            # ---- the whole batch in ONE call (unfz_run_batch) ------------------------------------------
            if has_reads:
                bind_blocks()
            b = L.Batch()
            b.sites = C.addressof(dsites.cols)
            b.reads = C.addressof(dreads.cols) if has_reads else None
            b.h_params = C.addressof(params)
            b.dnms, b.n_dnms, b.n_segs, b.segs, b.alleles = p_dnm, n, S, p_seg, p_all
            b.cap_pairs = int(caps["pairs"])
            b.seg_row_lo, b.seg_count, b.seg_pair_off = rp["seg_row_lo"], e1.ptr["seg_count"], z1.ptr["seg_pair_off"]
            b.scan_work, b.row_mark, b.mark_prefix = e1.ptr["scan_work"], z1.ptr["row_mark"], z1.ptr["mark_prefix"]
            b.guard, b.actual = z1.ptr["guard"], z1.ptr["guard"] + 64
            b.n_het, b.n_cand, b.cnv_dad, b.cnv_mom = rp["n_het"], rp["n_cand"], rp["cnv_dad"], rp["cnv_mom"]
            b.tally, b.calls_strict, b.calls_ambiguous, b.win = rp["tally"], rp["calls_s"], rp["calls_a"], rp["win"]
            b.cls, b.het_list, b.cand_list = e2.ptr["cls"], e2.ptr["het_list"], e2.ptr["cand_list"]
            b.cand_evid = z2.ptr["cand_evid"]
            if has_reads:
                b.max_l_seq, b.tile_reads, b.n_tiles = dreads.max_l_seq, tile_reads, n_tiles
                b.cap_hits = int(caps["hits"])
                for i_, v_ in enumerate(caps["chain"]):
                    b.cap_chain[i_] = int(v_)
                b.blk_maxspan, b.need, b.off = z1.ptr["blk_maxspan"], z1.ptr["need"], z1.ptr["off"]
                b.rsum = e1.ptr["rsum"]
                b.tile_tot, b.tile_base, b.tile_info = e1.ptr["tile_tot"], e1.ptr["tile_base"], e1.ptr["tile_info"]
                b.site_lo, b.site_n, b.seed_win = e2.ptr["site_lo"], e2.ptr["site_n"], e2.ptr["seed_win"]
                b.hits, b.scratch, b.scratch_bytes = e3.ptr["hits"], e3.ptr["scratch"], nbytes
                b.slot_label, b.slot_evid = z3.ptr["slot_label"], z3.ptr["slot_evid"]
                if want_ev:
                    b.ev_need, b.ev_off = z1.ptr["ev_need"], z1.ptr["ev_off"]
                    b.ev_read_dad, b.ev_read_mom = e3.ptr["ev_read_dad"], e3.ptr["ev_read_mom"]
                    b.ev_pos_dad, b.ev_pos_mom = e2.ptr["ev_pos_dad"], e2.ptr["ev_pos_mom"]
            if graph:
                zs = [z1, z2] + ([z3] if has_reads else [])
                spans = (L.Span * len(zs))(*[L.Span(z_.buf.data_ptr(), z_.buf.numel()) for z_ in zs])
                self._check(lib.unfz_run_batch_graph(ctx, C.byref(b), spans, len(zs), None, None, 0, s), "run_batch_graph")
            else:
                self._check(lib.unfz_run_batch(ctx, C.byref(b), s), "run_batch")
            launches += (22 if has_reads else 11) + (2 if want_ev else 0)
            h_pair_off, h_off = None, None
            res = BatchResult(plan=plan, n_pairs=int(caps["pairs"]), n_hits=int(caps["hits"]) if has_reads else 0,
                              seg_row_lo=None, seg_pair_off=None, n_het=None, n_cand=None, cnv_dad=None, cnv_mom=None)
            dv = res._dev
            dv.update(cls=e2.view["cls"], het_list=e2.view["het_list"].view(torch.int32),
                      cand_list=e2.view["cand_list"].view(torch.int32), cand_evid=z2.view["cand_evid"],
                      _keep=(z1, e1, z2, e2, d_plan))
            if has_reads:
                dv.update(rsum=e1.view["rsum"], hits=e3.view["hits"].view(torch.int32),
                          tile_base=e1.view["tile_base"].view(torch.int32), tile_reads=tile_reads,
                          slot_label=z3.view["slot_label"], slot_evid=z3.view["slot_evid"], row_mark=z1.view["row_mark"],
                          mark_prefix=z1.view["mark_prefix"].view(torch.int32), _keep3=(z3, e3))
        else:
            # ---- K0 + scan ---------------------------------------------------------------------
            self._check(lib.unfz_window_search(ctx, sc, p_seg, S, rp["seg_row_lo"], e1.ptr["seg_count"], s), "window_search")
            self._check(lib.unfz_exclusive_scan_i64(ctx, e1.ptr["seg_count"], z1.ptr["seg_pair_off"], S, e1.ptr["scan_work"], s), "scan(pairs)")
            launches += 4
            mark("window_search")
            guard_ptr, actual_ptr = z1.ptr["guard"], z1.ptr["guard"] + 64

            def check_caps(ptrs, limits, slot):
                k = len(ptrs)
                a_t = (C.c_void_p * k)(*ptrs)
                a_c = (C.c_int64 * k)(*[int(x) for x in limits])
                self._check(lib.unfz_check_caps(ctx, k, a_t, a_c, guard_ptr, actual_ptr + 8 * slot, s), "check_caps")

            h_pair_off = None
            if spec:
                lib.unfz_ctx_set_guard(ctx, guard_ptr)
                n_pairs = int(caps["pairs"])                                                 # capacity, not the total
                check_caps([z1.ptr["seg_pair_off"] + 8 * S], [n_pairs], 0)
                launches += 1
            else:
                h_pair_off = z1.view["seg_pair_off"].cpu().numpy().view(np.int64)[: S + 1]      # host sync 1
                n_pairs = int(h_pair_off[S]) if S > 0 else 0

            if not spec:
                z2, e2 = arena2(n_pairs)
            mark("alloc1")
            self._check(lib.unfz_classify_sites(ctx, sc, p_seg, rp["seg_row_lo"], z1.ptr["seg_pair_off"], S, n_pairs,
                                                C.byref(params), e2.ptr["cls"], s), "classify_sites")
            launches += 1 if n_pairs else 0
            mark("classify_sites")
            self._check(lib.unfz_compact_sites(ctx, p_dnm, n, p_seg, rp["seg_row_lo"], z1.ptr["seg_pair_off"], e2.ptr["cls"],
                                               e2.ptr["het_list"], rp["n_het"], e2.ptr["cand_list"], rp["n_cand"], rp["cnv_dad"],
                                               rp["cnv_mom"], z1.ptr["row_mark"], s), "compact_sites")
            self._check(lib.unfz_exclusive_scan_u8_i32(ctx, z1.ptr["row_mark"], z1.ptr["mark_prefix"], V, e1.ptr["scan_work"], s), "scan(marks)")
            launches += 4
            mark("compact_sites")

            res = BatchResult(plan=plan, n_pairs=n_pairs, n_hits=0, seg_row_lo=None, seg_pair_off=h_pair_off,
                              n_het=None, n_cand=None, cnv_dad=None, cnv_mom=None)
            dv = res._dev
            dv.update(cls=e2.view["cls"], het_list=e2.view["het_list"].view(torch.int32), cand_list=e2.view["cand_list"].view(torch.int32),
                      cand_evid=z2.view["cand_evid"], _keep=(z1, e1, z2, e2, d_plan))

            if has_reads:
                rc_ = C.byref(dreads.cols)
                bind_blocks()
                # ---- K2 + scan(tile hit totals) + chain sizing; ONE host sync for all the sizes ------------
                off_ptr = z1.ptr["off"]
                total_hits_ptr = off_ptr + 8 * 6 * (n + 1)
                mark("alloc2")
                self._check(lib.unfz_read_scan(ctx, rc_, sc, z1.ptr["mark_prefix"], C.byref(params), dreads.max_l_seq, e1.ptr["rsum"],
                                               z1.ptr["blk_maxspan"], e1.ptr["tile_tot"], e1.ptr["tile_info"], s),
                            "read_scan")
                launches += 1
                mark("read_scan")
                self._check(lib.unfz_exclusive_scan_u32(ctx, e1.ptr["tile_tot"], e1.ptr["tile_base"], n_tiles, total_hits_ptr,
                                                        e1.ptr["scan_work"], s), "scan(hits)")
                launches += 3
                mark("scan_hits")
                self._check(lib.unfz_chain_size(ctx, p_dnm, n, p_seg, z1.ptr["seg_pair_off"], sc, rc_, e1.ptr["rsum"],
                                                z1.ptr["blk_maxspan"], e2.ptr["het_list"], rp["n_het"], e2.ptr["cand_list"],
                                                rp["n_cand"], rp["win"], z1.ptr["need"], e2.ptr["site_lo"], e2.ptr["site_n"],
                                                e2.ptr["seed_win"], s), "chain_size")
                self._check(lib.unfz_exclusive_scan_rows_i64(ctx, z1.ptr["need"], off_ptr, 6, n, s), "scan(need)")
                launches += 2
                h_off = None
                if spec:
                    totals = np.asarray(caps["chain"], dtype=np.int64).copy()
                    n_hits = int(caps["hits"])
                    check_caps([off_ptr + 8 * ((i + 1) * (n + 1) - 1) for i in range(6)] + [total_hits_ptr],
                               list(totals) + [n_hits], 1)
                    launches += 1
                else:
                    h_all = z1.view["off"].cpu().numpy().view(np.int64)                      # host sync 2
                    h_off = h_all[: 6 * (n + 1)].reshape(6, n + 1)
                    n_hits = int(h_all[6 * (n + 1)])
                    totals = np.ascontiguousarray(h_off[:, n]).astype(np.int64)
                mark("chain_size")
                if n_hits >= 2**32:
                    raise RuntimeError("more than 2^32 read x site hits in one batch")
                res.n_hits = n_hits
                if not spec:
                    z3, e3, nbytes = arena3(totals, n_hits)
                mark("alloc3")
                self._check(lib.unfz_read_site_alleles(ctx, rc_, sc, z1.ptr["row_mark"], z1.ptr["mark_prefix"], e1.ptr["rsum"],
                                                       e1.ptr["tile_base"], tile_reads, e3.ptr["hits"],
                                                       e1.ptr["tile_info"], s),
                            "read_site_alleles")
                launches += 1
                mark("read_site_alleles")
                self._check(lib.unfz_chain_tally(ctx, p_dnm, n, p_seg, z1.ptr["seg_pair_off"], sc, rc_, e1.ptr["rsum"],
                                                 z1.ptr["blk_maxspan"], e3.ptr["hits"], e1.ptr["tile_base"], tile_reads, z1.ptr["mark_prefix"],
                                                 e2.ptr["het_list"],
                                                 rp["n_het"], e2.ptr["cand_list"], rp["n_cand"], p_all, rp["win"], e2.ptr["site_lo"], e2.ptr["site_n"],
                                                 e2.ptr["seed_win"], off_ptr,
                                                 totals.ctypes.data, C.byref(params), e3.ptr["scratch"], nbytes,
                                                 z3.ptr["slot_label"], z3.ptr["slot_evid"], z2.ptr["cand_evid"], rp["tally"],
                                                 z1.ptr["ev_need"] if want_ev else None, s),
                            "chain_tally")
                launches += 3
                mark("chain_tally")
                if want_ev:
                    self._check(lib.unfz_exclusive_scan_rows_i64(ctx, z1.ptr["ev_need"], z1.ptr["ev_off"], 4, n, s), "scan(ev)")
                    self._check(lib.unfz_evidence_lists(ctx, p_dnm, n, z1.ptr["seg_pair_off"], sc, e2.ptr["cand_list"], rp["n_cand"],
                                                        z2.ptr["cand_evid"], rp["win"], off_ptr, z3.ptr["slot_evid"], z1.ptr["ev_off"],
                                                        e3.ptr["ev_read_dad"], e3.ptr["ev_read_mom"], e2.ptr["ev_pos_dad"],
                                                        e2.ptr["ev_pos_mom"], s),
                                "evidence_lists")
                    launches += 2
                    mark("evidence_lists")
                dv.update(rsum=e1.view["rsum"], hits=e3.view["hits"].view(torch.int32),
                          tile_base=e1.view["tile_base"].view(torch.int32), tile_reads=tile_reads, slot_label=z3.view["slot_label"],
                          slot_evid=z3.view["slot_evid"], row_mark=z1.view["row_mark"],
                          mark_prefix=z1.view["mark_prefix"].view(torch.int32), _keep3=(z3, e3))
                if h_off is not None:
                    res.slot_off = h_off[0].copy()
            self._check(lib.unfz_summarize(ctx, p_dnm, n, rp["tally"], rp["cnv_dad"], rp["cnv_mom"], rp["n_cand"], C.byref(params),
                                           rp["calls_s"], rp["calls_a"], s), "summarize")
            launches += 1
            mark("summarize")
        # ---- results: ONE device-to-host copy of the int32 result block ----------------------------
        if spec:
            lib.unfz_ctx_set_guard(ctx, None)
        front_buf, done = None, None
        if download:
            # pinned target (a pageable D2H copy is several times slower and serialises with the driver).  With recycled
            # arenas the pinned block rotates with them: allocating pinned memory is a slow, device-synchronising call
            # (tens of milliseconds on an 8-GPU box), so a steady-state batch must not make one; the result arrays are
            # then copied out of the block in finish(), before the set is handed back
            pkey = ("pinned", int(dl_end))
            q_ = pool.get(pkey) if reuse else None
            front_buf = q_.popleft() if q_ else torch.empty((dl_end,), dtype=torch.uint8, pin_memory=True)
            front_buf.copy_(z1.buf[:dl_end], non_blocking=True)
            done = torch.cuda.Event()
            done.record(st)

        def finish():
            nonlocal res
            if download:
                done.synchronize()
                front = front_buf.numpy().copy() if reuse else front_buf.numpy()
                self.last_d2h_bytes = int(dl_end)
                item = {nm: (off, nb) for nm, off, nb in z1.items}
                sect = lambda nm: front[item[nm][0]: item[nm][0] + item[nm][1]]
                hr = sect("result").view(np.int32)
                if spec:
                    g_ = sect("guard")
                    actual = g_[64: 64 + 64].view(np.int64)
                    if int(g_[:4].view(np.int32)[0]) != 0:
                        # a capacity was exceeded: nothing was written out of bounds, run again with exact sizes
                        self.spec_fallbacks += 1
                        self._caps = None
                        dv.clear()
                        return self.run(dsites, dreads, plan, params, blk_cul=blk_cul, time_stages=time_stages,
                                        download=download, keep_device=keep_device, speculative=False, evidence=evidence)
                    res.seg_pair_off = sect("seg_pair_off").view(np.int64)[: S + 1].copy()
                    res.n_pairs = int(actual[0])
                    if has_reads:
                        o0 = item["off"][0]
                        res.slot_off = front[o0: o0 + 8 * (n + 1)].view(np.int64).copy()
                        res.n_hits = int(actual[7])
                        chain_now = [int(x) for x in actual[1:7]]
                elif has_reads:
                    chain_now = [int(x) for x in h_off[:, n]]
                # capacities for the next batch: what this one needed, plus a quarter
                need_now = {"pairs": res.n_pairs, "hits": res.n_hits, "chain": chain_now if has_reads else [0] * 6}
                grow = lambda v: int(v * 1.25) + 4096
                cur = getattr(self, "_caps", None)
                if cur is None:
                    self._caps = {"pairs": grow(need_now["pairs"]), "hits": grow(need_now["hits"]),
                                  "chain": [grow(v) for v in need_now["chain"]]}
                else:
                    cur["pairs"] = max(cur["pairs"], grow(need_now["pairs"]) if need_now["pairs"] > 0.9 * cur["pairs"] else 0)
                    cur["hits"] = max(cur["hits"], grow(need_now["hits"]) if need_now["hits"] > 0.9 * cur["hits"] else 0)
                    cur["chain"] = [max(c, grow(v) if v > 0.9 * c else 0) for c, v in zip(cur["chain"], need_now["chain"])]
                g = lambda nm, cnt: hr[r_off[nm]: r_off[nm] + cnt]
                res.seg_row_lo = g("seg_row_lo", S)
                res.n_het, res.n_cand = g("n_het", n), g("n_cand", n)
                res.cnv_dad, res.cnv_mom = g("cnv_dad", n), g("cnv_mom", n)
                res.tally = g("tally", 8 * n).view(L.TALLY_DTYPE)
                res.calls_strict = g("calls_s", 4 * n).view(L.CALL_DTYPE)
                res.calls_ambiguous = g("calls_a", 4 * n).view(L.CALL_DTYPE)
                res.win = g("win", 4 * n).reshape(4, n)
                if want_ev:
                    # second, small download: the evidence lists, now that their lengths are on the host.  It goes over
                    # the side stream: behind a deferred batch the main stream may already hold the next batch's copies
                    eo = sect("ev_off").view(np.int64).reshape(4, n + 1).copy()
                    tot = [int(eo[q, n]) for q in range(4)]
                    parts = [(e3.view["ev_read_dad"], 4 * tot[0]), (e3.view["ev_read_mom"], 4 * tot[1]),
                             (e2.view["ev_pos_dad"], 4 * tot[2]), (e2.view["ev_pos_mom"], 4 * tot[3])]
                    # pinned blocks come from the engine's own size-class lists (no pinned allocation in steady state,
                    # see above) and go back as soon as the lists are copied out
                    bufs, blocks = [], []
                    with torch.cuda.stream(self.stream2):
                        for t_, nb_ in parts:
                            hb = self._pinned_block(nb_)
                            if nb_:
                                hb[:nb_].copy_(t_[:nb_], non_blocking=True)
                            blocks.append(hb)
                    self.stream2.synchronize()
                    for hb, (t_, nb_) in zip(blocks, parts):
                        bufs.append(hb.numpy()[:nb_].copy().view(np.int32))
                        self._pinned_free.setdefault(int(hb.numel()), []).append(hb)
                    res.ev = {"off": eo, "read_dad": bufs[0], "read_mom": bufs[1], "pos_dad": bufs[2], "pos_mom": bufs[3]}
                    self.last_d2h_bytes += 4 * sum(tot)
            mark("download")
            res.launches = launches
            if time_stages:
                torch.cuda.synchronize(dev)
                for (n0, e0), (n1, e1_) in zip(ev[:-1], ev[1:]):
                    res.timings_ms[n1] = res.timings_ms.get(n1, 0.0) + e0.elapsed_time(e1_)
            if not keep_device:
                dv.clear()
                # stale layouts are dropped by size, not by count: a few batches in flight times six arenas is dozens of
                # live buffers, and clearing them mid-stream would cost every batch a fresh allocation and graph
                if len(pool) > 48 or sum(b_.numel() for q_ in pool.values() for b_ in q_) > self._pool_limit:
                    pool.clear()
                for a_ in arenas:
                    pool.setdefault(a_.key, collections.deque()).append(a_.buf)
                if download and reuse:
                    pool.setdefault(pkey, collections.deque()).append(front_buf)
            return res

        if defer:
            if time_stages or not download:
                raise ValueError("defer=True needs download=True and no stage timers")
            return PendingBatch(finish)
        return finish()
