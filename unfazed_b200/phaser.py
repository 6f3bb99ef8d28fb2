"""Batch phasing over columnar tables: plan -> engine -> the reference's record dicts.

This is the host-side mirror of ``snv_phaser.run_read_phasing`` (reference :206-299),
``sv_phaser.phase_svs`` (:427-493) and ``informative_site_finder.find`` (:167-344) for a whole DNM
list at once.  All arithmetic happens in the CUDA kernels; this file only plans windows and
reshapes results.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import numpy as np

from . import _lib as L
from . import _records            # csrc/records.c, built in-tree by csrc/Makefile (no Python fallback)
from .engine import BatchResult, DeviceReads, DeviceSites, Engine, PackedReads, make_params
from .plan import (SNV_TYPES, SV_TYPES, Plan, SiteIndex, concat_plans, concordant_upper_lens,
                   plan_find_fast)
from .schema import ReadTable, SiteTable, min_base_qual


def dnm_key(dn: dict) -> str:
    """records key, snv_phaser.py:202."""
    return "_".join([str(dn["chrom"]), str(dn["start"]), str(dn["end"]), dn["kid"], dn["vartype"]])


class CompactRecords:
    """The records of one shard before they are Python dicts: the live DNM entries plus the flat evidence lists they are
    cut from.  This is what a rank sends to rank 0 in a multi-GPU run -- a few numpy arrays pickle and unpickle in
    microseconds, whereas unpickling the finished dicts (hundreds of thousands of small strings) made rank 0 the serial
    bottleneck of the cohort job.  ``to_records()`` is the same native builder ``BatchPhaser.records`` uses."""

    def __init__(self, entries, ped, auto, names, pair_ids, n_read_dad, pos_dad, pos_mom, off):
        self.entries, self.ped, self.auto = entries, ped, auto
        self.names, self.pair_ids, self.n_read_dad = names, pair_ids, int(n_read_dad)
        self.pos_dad, self.pos_mom, self.off = pos_dad, pos_mom, off

    def __len__(self):
        return len(self.entries)

    def to_records(self, out: Optional[Dict[str, dict]] = None) -> Dict[str, dict]:
        import gc
        out = {} if out is None else out
        was_on = gc.isenabled()
        gc.disable()                    # thousands of small containers, no cycles: a collection in the middle only costs time
        try:
            return self._to_records(out)
        finally:
            if was_on:
                gc.enable()

    def _to_records(self, out: Dict[str, dict]) -> Dict[str, dict]:
        k = len(self.entries)
        n_r = len(self.names) if self.names is not None else int(self.pair_ids.shape[0])
        idx = np.arange(n_r, dtype=np.int32)
        _records.read_records(out, self.entries, self.ped, np.arange(k, dtype=np.int64), np.ascontiguousarray(self.auto, dtype=np.uint8),
                              self.names, self.pair_ids, idx[: self.n_read_dad], idx[self.n_read_dad:],
                              np.ascontiguousarray(self.pos_dad, dtype=np.int32), np.ascontiguousarray(self.pos_mom, dtype=np.int32),
                              np.ascontiguousarray(self.off, dtype=np.int64))
        return out


def _cut(flat: np.ndarray, off: np.ndarray, live: np.ndarray):
    """The slices flat[off[d]:off[d+1]] of the entries in ``live``, concatenated, and their new offsets."""
    lens = off[live + 1] - off[live]
    new_off = np.zeros(live.shape[0] + 1, dtype=np.int64)
    np.cumsum(lens, out=new_off[1:])
    tot = int(new_off[-1])
    if tot == int(flat.shape[0]):                    # entries without a record own no evidence: nothing to drop
        return flat, new_off
    src = np.repeat(off[live] - new_off[:-1], lens) + np.arange(tot, dtype=np.int64)
    return flat[src], new_off


class BatchPhaser:
    """``resident=True`` (default): the site and read columns are uploaded once and stay in HBM across
    calls.  ``resident=False``: every call copies them from the host arrays it was given (pinned
    arrays copy asynchronously) and releases them afterwards -- the end-to-end mode of ``bench.py``.
    ``reads`` is a ReadTable or an engine.PackedReads (the columns as they cross PCIe)."""

    def __init__(self, engine: Engine, sites: SiteTable, reads, pedigrees: dict,
                 dsites: Optional[DeviceSites] = None, dreads: Optional[DeviceReads] = None, resident: bool = True):
        self.engine = engine
        self.packed = reads if isinstance(reads, PackedReads) else None
        self.sites, self.reads, self.ped = sites, (reads.table if self.packed is not None else reads), pedigrees
        self.sidx = SiteIndex(sites)
        self.resident = resident
        self._dsites = dsites
        # the read columns go up with the low-quality plane of one --min-gt-qual: uploaded at first use
        self._dreads = dreads
        self._cul_cache: Dict[tuple, np.ndarray] = {}
        self.last_timing: Dict[str, float] = {}

    # -------------------------------------------------------------------------------------
    @property
    def dsites(self) -> DeviceSites:
        if self._dsites is None:
            self._dsites = self.engine.upload_sites(self.sites)
        return self._dsites

    def dreads_for(self, min_gt_qual=20) -> Optional[DeviceReads]:
        if self.reads is None:
            return None
        mb = min_base_qual(min_gt_qual)
        if self._dreads is None or self._dreads.min_bq != mb:
            self._dreads = None                      # release the old planes first
            if self.reads.qual is None:
                # decoded on the device: the planes of this threshold are emitted again from the resident records
                self._dreads = self.reads.device_source.device_reads(min_gt_qual)
                return self._dreads
            src = self.packed if (self.packed is not None and self.packed.min_bq == mb) else self.reads
            self._dreads = self.engine.upload_reads(src, min_gt_qual=min_gt_qual)
        return self._dreads

    @property
    def dreads(self) -> Optional[DeviceReads]:
        return self._dreads if self._dreads is not None else self.dreads_for(20)

    def release_device(self):
        self._dsites = None
        self._dreads = None

    def cul(self, readlen, insert_size_max_sample, stdevs) -> Optional[np.ndarray]:
        if self.reads is None:
            return None
        key = (readlen, insert_size_max_sample, stdevs)
        if key not in self._cul_cache:
            self._cul_cache[key] = self.engine.concordant_upper_lens(self.dreads, readlen, insert_size_max_sample, stdevs)
        return self._cul_cache[key]

    def site_dicts(self, res: BatchResult, d: int, trio: int, with_kid_allele: bool):
        """candidate_sites / het_sites of entry d in the reference's dict form."""
        s = self.sites
        kid, dad, mom = s.trios[trio]
        hets = [{"pos": int(s.pos[r]), "ref_allele": chr(s.ref[r]), "alt_allele": chr(s.alt[r])}
                for r in res.het_rows(d).tolist()]
        cands = []
        for w in res.cand_words(d).view(np.uint32).tolist():
            r = w & 0x3FFFFFFF
            c = {"pos": int(s.pos[r]), "ref_allele": chr(s.ref[r]), "alt_allele": chr(s.alt[r])}
            if with_kid_allele:
                c["kid_allele"] = "alt_parent" if (w & 0x40000000) else "ref_parent"
            if w & 0x80000000:
                c["alt_parent"], c["ref_parent"] = dad, mom
            else:
                c["alt_parent"], c["ref_parent"] = mom, dad
            cands.append(c)
        return cands, hets

    # -------------------------------------------------------------------------------------
    def plan_batch(self, snvs: List[dict], svs: List[dict], *, threads=2, build="38", multiread_proc_min=1000,
                   search_dist=5000):
        """Window plan of one call: the CNV entries of the SVs (find with search_dist 0, whole region:
        sv_phaser.py:375-389), the read entries of the SVs, the read entries of the SNVs.  Returns
        (plan, layout) where layout gives the three entry ranges."""
        common = dict(build=build, multiread_proc_min=multiread_proc_min, threads=threads)
        plans: List[Plan] = []
        n0 = 0
        a0 = 0

        def add(dnms, **kw):
            nonlocal n0, a0
            p = plan_find_fast(dnms, self.ped, self.sidx, self.reads, first_entry=n0, alleles_base=a0, **common, **kw)
            plans.append(p)
            n0 += len(dnms)
            a0 += int(p.alleles.shape[0])
            return p

        layout = {"sv_cnv": (0, 0), "sv_read": (0, 0), "snv": (0, 0)}
        if svs:
            add(svs, search_dist=0, whole_region=True, with_reads=False)
            layout["sv_cnv"] = (0, len(svs))
            p = add(svs, search_dist=search_dist, whole_region=False, with_reads=True, sv_quirk=True)
            p.dnm["cnv_entry"] = np.arange(len(svs), dtype=np.int32)
            layout["sv_read"] = (len(svs), 2 * len(svs))
        if snvs:
            add(snvs, search_dist=search_dist, whole_region=False, with_reads=True)
            layout["snv"] = (n0 - len(snvs), n0)
        return concat_plans(plans), layout

    def run(self, snvs: List[dict], svs: List[dict], *, threads=2, build="38", no_extended=False,
            multiread_proc_min=1000, ab_homref=(0.0, 0.2), ab_homalt=(0.8, 1.0), ab_het=(0.2, 0.8),
            min_gt_qual=20, min_depth=10, search_dist=5000, insert_size_max_sample=1000000, stdevs=3,
            min_map_qual=1, readlen=151, split_error_margin=5, evidence_min_ratio=10,
            time_stages=False, evidence=True, keep_device=True, defer=False):
        """Plan + run all entries of one call.  Returns (result, layout); with ``defer`` the first element is an
        engine.PendingBatch whose ``finish()`` gives the result (see ``phase_stream``)."""
        import time as _t
        t0 = _t.perf_counter()
        if not self.resident:
            # the copies are asynchronous when the host arrays are pinned: the windows are planned while they fly
            self.release_device()
            _ = self.dsites
            self.dreads_for(min_gt_qual)
        t1 = _t.perf_counter()
        plan, layout = self.plan_batch(snvs, svs, threads=threads, build=build, multiread_proc_min=multiread_proc_min,
                                       search_dist=search_dist)
        t2 = _t.perf_counter()
        params = make_params(ab_homref, ab_homalt, ab_het, min_gt_qual, min_depth, min_map_qual, readlen,
                             insert_size_max_sample, no_extended, evidence_min_ratio, split_error_margin)
        dreads = self.dreads_for(min_gt_qual)
        res = self.engine.run(self.dsites, dreads, plan, params,
                              blk_cul=self.cul(readlen, insert_size_max_sample, stdevs), time_stages=time_stages,
                              evidence=evidence, keep_device=keep_device, defer=defer)
        t3 = _t.perf_counter()
        if not self.resident:
            self.release_device()
        self.last_timing = {"issue_uploads_ms": (t1 - t0) * 1e3, "plan_ms": (t2 - t1) * 1e3,
                            "run_until_results_ms": (t3 - t2) * 1e3}
        return res, layout

    # -------------------------------------------------------------------------------------
    def _read_record(self, res: BatchResult, d: int, dn: dict):
        kid = dn["kid"]
        dad, mom = self.ped[kid]["dad"], self.ped[kid]["mom"]
        s = self.sites
        ev = res.cand_evidence(d)
        rows = res.cand_words(d).view(np.uint32) & 0x3FFFFFFF
        pos = s.pos[rows.astype(np.int64)]
        dad_sites = sorted({str(int(p)) for p, e in zip(pos, ev) if e & 1})
        mom_sites = sorted({str(int(p)) for p, e in zip(pos, ev) if e & 2})
        sev = res.slot_evidence(d)
        nm = self.reads.name_of
        dad_reads = sorted({nm(int(r)) for r in res.slot_reads(d, np.nonzero(sev & 1)[0])})
        mom_reads = sorted({nm(int(r)) for r in res.slot_reads(d, np.nonzero(sev & 2)[0])})
        return {
            "region": {"chrom": dn["chrom"], "start": dn["start"], "end": dn["end"]},
            "vartype": dn["vartype"], "kid": kid, "dad": dad, "mom": mom,
            "dad_sites": dad_sites, "mom_sites": mom_sites, "evidence_type": "readbacked",
            "dad_reads": dad_reads, "mom_reads": mom_reads,
            "cnv_dad_sites": "", "cnv_mom_sites": "", "cnv_evidence_type": "",
        }

    @staticmethod
    def _auto_record(dn, dad, mom):
        return {
            "region": {"chrom": dn["chrom"], "start": dn["start"], "end": dn["end"]},
            "vartype": dn["vartype"], "kid": dn["kid"], "dad": dad, "mom": mom,
            "cnv_dad_sites": "NA", "cnv_mom_sites": "NA", "cnv_evidence_type": "SEX-CHROM",
            "dad_sites": "", "mom_sites": "", "evidence_type": "SEX-CHROM",
            "dad_reads": [], "mom_reads": [],
        }

    def records(self, res: BatchResult, layout) -> Dict[str, dict]:
        """The dict ``phase_snvs``/``phase_svs`` return, merged as unfazed.py:648-649 does."""
        # tens of thousands of small containers are created below; a cyclic-GC pass in the middle only costs time
        # (nothing here can form a cycle), so the collector is paused for the duration of the call
        import gc
        was_on = gc.isenabled()
        gc.disable()
        try:
            return self._records(res, layout)
        finally:
            if was_on:
                gc.enable()

    def _records(self, res: BatchResult, layout) -> Dict[str, dict]:
        plan = res.plan
        out_sv: Dict[str, dict] = {}
        out_snv: Dict[str, dict] = {}
        s = self.sites
        a, b = layout["sv_cnv"]
        cnv: Dict[str, dict] = {}
        if b > a:
            # phase_by_snvs (sv_phaser.py:71-85) for all CNV entries at once: every candidate votes for
            # site[site["kid_allele"]]; the per-parent str(pos) lists are cut out of two flat lists
            n_c = np.asarray(res.n_cand[a:b], dtype=np.int64)
            seg_lo, seg_hi = plan.dnm["seg_lo"][a:b], plan.dnm["seg_hi"][a:b]
            base = np.where(seg_hi > seg_lo, res.seg_pair_off[np.minimum(seg_lo, len(res.seg_pair_off) - 1)], 0).astype(np.int64)
            is_cnv = np.fromiter((plan.entries[d]["vartype"] in ("DEL", "DUP") for d in range(a, b)), dtype=bool, count=b - a)
            n_c = np.where(is_cnv, n_c, 0)
            tot = int(n_c.sum())
            if tot:
                owner = np.repeat(np.arange(b - a), n_c)
                flat = np.repeat(base, n_c) + (np.arange(tot) - np.repeat(np.cumsum(n_c) - n_c, n_c))
                w = res._np("cand_list").view(np.uint32)[flat]
                dad_vote = ((w >> 31) & 1) == ((w >> 30) & 1)
                strs = np.array(list(map(str, s.pos[(w & 0x3FFFFFFF).astype(np.int64)].tolist())), dtype=object)
                d_flat, m_flat = strs[dad_vote].tolist(), strs[~dad_vote].tolist()
                nd_ = np.bincount(owner[dad_vote], minlength=b - a)
                od = np.concatenate([[0], np.cumsum(nd_)]).tolist()
                om = np.concatenate([[0], np.cumsum(n_c - nd_)]).tolist()
            flags_c = plan.dnm["flags"][a:b].tolist()
            n_cl = n_c.tolist()
            for i, d in enumerate(range(a, b)):
                dn = plan.entries[d]
                dad, mom = self.ped[dn["kid"]]["dad"], self.ped[dn["kid"]]["mom"]
                if flags_c[i] & L.DNM_AUTOPHASE:
                    cnv[dnm_key(dn)] = self._auto_record(dn, dad, mom)
                    continue
                if n_cl[i] == 0:
                    continue
                cnv[dnm_key(dn)] = {
                    "region": {"chrom": dn["chrom"], "start": dn["start"], "end": dn["end"]},
                    "vartype": dn["vartype"], "kid": dn["kid"], "dad": dad, "mom": mom,
                    "cnv_dad_sites": d_flat[od[i]:od[i + 1]], "cnv_mom_sites": m_flat[om[i]:om[i + 1]],
                    "cnv_evidence_type": "ALLELE-BALANCE",
                    "dad_sites": "", "mom_sites": "", "evidence_type": "", "dad_reads": [], "mom_reads": [],
                }
        ev = res.ev
        flags_a = plan.dnm["flags"]
        has_a = res.tally["has_record"] if res.tally is not None else np.zeros(len(flags_a), dtype=np.int32)
        ped = self.ped
        entries = plan.entries
        for name, out in (("sv_read", out_sv), ("snv", out_snv)):
            a, b = layout[name]
            # only the entries that get a record are visited (in entry order): autophased ones and those with matches
            live = a + np.flatnonzero(((flags_a[a:b] & L.DNM_AUTOPHASE) != 0) | (has_a[a:b] != 0))
            auto = (flags_a[live] & L.DNM_AUTOPHASE) != 0
            if ev is not None:
                # evidence lists compacted per DNM and per parent on the device (evidence_lists_kernel): the native builder
                # (csrc/records.c) cuts every record out of the four flat lists.  One pair = one window slot = one name, so
                # the read lists are unique as they come (slot order); a site seen through two overlapping windows (Q9)
                # appears twice, the reference keeps a set of str(pos) -> sorted(set(...)) there too
                names = self.reads.names
                if names is not None and not isinstance(names, list):
                    names = self.reads.names = list(names)
                _records.read_records(out, entries, ped, np.ascontiguousarray(live, dtype=np.int64),
                                      np.ascontiguousarray(auto, dtype=np.uint8), names,
                                      None if names is not None else np.ascontiguousarray(self.reads.pair_ids(), dtype=np.int64),
                                      ev["read_dad"], ev["read_mom"], ev["pos_dad"], ev["pos_mom"],
                                      np.ascontiguousarray(ev["off"], dtype=np.int64))
                continue
            for d, is_auto in zip(live.tolist(), auto.tolist()):
                dn = entries[d]
                p = ped[dn["kid"]]
                out[dnm_key(dn)] = self._auto_record(dn, p["dad"], p["mom"]) if is_auto else self._read_record(res, d, dn)
        for k, c in cnv.items():                                  # sv_phaser.py:484-492
            if k not in out_sv:
                out_sv[k] = c
            else:
                out_sv[k]["cnv_dad_sites"] = c["cnv_dad_sites"]
                out_sv[k]["cnv_mom_sites"] = c["cnv_mom_sites"]
                out_sv[k]["evidence_type"] += "," + c["cnv_evidence_type"]
        out_snv.update(out_sv)
        return out_snv

    def compact(self, res: BatchResult, layout) -> Optional[CompactRecords]:
        """The records of a batch in compact form (see CompactRecords), or None when the batch needs the general path
        (SV entries merge CNV votes into their records; runs without device evidence lists)."""
        if res.ev is None or layout["sv_cnv"][1] > layout["sv_cnv"][0] or layout["sv_read"][1] > layout["sv_read"][0]:
            return None
        plan, ev = res.plan, res.ev
        a, b = layout["snv"]
        flags_a = plan.dnm["flags"]
        has_a = res.tally["has_record"] if res.tally is not None else np.zeros(len(flags_a), dtype=np.int32)
        live = a + np.flatnonzero(((flags_a[a:b] & L.DNM_AUTOPHASE) != 0) | (has_a[a:b] != 0))
        auto = ((flags_a[live] & L.DNM_AUTOPHASE) != 0).astype(np.uint8)
        entries = [plan.entries[d] for d in live.tolist()]
        entries = [{"chrom": e["chrom"], "start": e["start"], "end": e["end"], "kid": e["kid"], "vartype": e["vartype"]} for e in entries]
        ped = {k: {"dad": self.ped[k]["dad"], "mom": self.ped[k]["mom"]} for k in {e["kid"] for e in entries}}
        off = np.asarray(ev["off"], dtype=np.int64)
        rd, o_rd = _cut(ev["read_dad"], off[0], live)
        rm, o_rm = _cut(ev["read_mom"], off[1], live)
        pd_, o_pd = _cut(ev["pos_dad"], off[2], live)
        pm_, o_pm = _cut(ev["pos_mom"], off[3], live)
        ridx = np.concatenate([rd, rm]).astype(np.int64)
        if self.reads.names is not None:
            nm = self.reads.names
            names, pair_ids = [nm[i] for i in ridx.tolist()], None
        else:
            names, pair_ids = None, np.ascontiguousarray(self.reads.pair_ids()[ridx], dtype=np.int64)
        o_rm = o_rm                                             # offsets of the mom lists index the second half
        return CompactRecords(entries, ped, auto, names, pair_ids, rd.shape[0], np.array(pd_, dtype=np.int32),
                              np.array(pm_, dtype=np.int32), np.stack([o_rd, o_rm, o_pd, o_pm]))

    def labels(self, res: BatchResult, d: int) -> Dict[str, str]:
        """read name -> haplotype ('ref' | 'alt' | 'ref+alt') of entry d (parity checks)."""
        lab = res.slot_labels(d)
        names = {1: "ref", 2: "alt", 3: "ref+alt"}
        xs = np.nonzero(lab)[0]
        return {self.reads.name_of(int(r)): names[int(lab[x])] for x, r in zip(xs, res.slot_reads(d, xs))}

    def _split(self, dnms: List[dict]):
        kids = set(self.ped)
        svs = [d for d in dnms if d["vartype"].upper() in SV_TYPES and d["kid"] in kids]
        snvs = [d for d in dnms if d["vartype"].upper() in SNV_TYPES and d["kid"] in kids]
        return snvs, svs

    def _deliver(self, res: BatchResult, layout, compact: bool):
        if compact:
            c = self.compact(res, layout)
            if c is not None:
                return c
        return self.records(res, layout)

    def phase(self, dnms: List[dict], compact: bool = False, **params):
        """DNM dicts in, the record dict of phase_snvs/phase_svs out.  ``compact=True`` returns a CompactRecords when the
        batch allows it (what a rank ships to rank 0 in a multi-GPU run; ``.to_records()`` gives the same dict)."""
        import time as _t
        snvs, svs = self._split(dnms)
        # the CNV votes of SVs are read from the device lists while the records are built; otherwise nothing has to
        # stay on the device and the engine recycles its buffers (and replays the batch as a CUDA graph)
        res, layout = self.run(snvs, svs, keep_device=bool(svs), **params)
        t0 = _t.perf_counter()
        out = self._deliver(res, layout, compact)
        self.last_timing["records_ms"] = (_t.perf_counter() - t0) * 1e3
        return out

    def phase_stream(self, batches, compact: bool = False, **params):
        """Phase a sequence of DNM lists, yielding one record dict per list, in order.  Software pipeline of depth two:
        the copies and kernels of list k+1 are put on the stream BEFORE the host waits for list k and turns its
        results into record dicts, so host work (about half of an end-to-end step) and PCIe/GPU work overlap."""
        import time as _t
        pending = None

        def finish(p):
            t0 = _t.perf_counter()
            res = p[0].finish()
            t1 = _t.perf_counter()
            out = self._deliver(res, p[1], compact)
            self.last_timing.update(wait_results_ms=(t1 - t0) * 1e3, records_ms=(_t.perf_counter() - t1) * 1e3)
            return out

        for dnms in batches:
            snvs, svs = self._split(dnms)
            h, layout = self.run(snvs, svs, keep_device=bool(svs), defer=True, **params)
            if pending is not None:
                yield finish(pending)
            pending = (h, layout)
        if pending is not None:
            yield finish(pending)
