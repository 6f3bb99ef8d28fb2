"""Where the drop-in modules get their columnar tables from.

* ``*.npz`` written by ``tableio.save_tables`` (our native cache of decoded inputs), or
* indexed BAM files (``*.bam`` with a ``.bai``) through ``bamio.py``, natively -- no pysam needed, and with an
  engine the bulk of the records is decoded on the GPU, or
* indexed BAM files (``*.bam`` with a ``.bai`` or ``.csi``) through ``bamio.py`` as above, or
* CRAM 3.0 files with a ``.crai`` and a plain-text FASTA reference through ``cramio.py``, decoded to the BAM records
  ``bamio.py`` reads, or
* a bgzipped, indexed sites VCF (``*.vcf.gz`` / ``*.vcf.bgz`` with a ``.tbi`` or ``.csi``) through ``vcfio.py``, natively
  -- no cyvcf2 needed, and with an engine the genotype fields are decoded on the GPU, or
* a CSI-indexed BCF 2.2 sites file (``*.bcf`` with a ``.csi``) through ``bcfio.py``, natively, likewise, or
* other sites VCF/BCF files (unindexed, uncompressed BCF, other BCF versions) through ``cyvcf2`` and the kids' other alignment files (other CRAM versions, unindexed CRAM or BAM) through ``pysam``
  -- imported lazily, so the package works without them as long as tables are supplied -- decoded only around
  the DNMs and packed by ``packers.py``.

Tables are cached per (file, request) for the lifetime of the process, like the reference's
``concordant_upper_lens`` cache (snv_phaser.py:14).
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional, Tuple

import numpy as np

from . import bamio, bcfio, cramio, packers, vcfio
from .plan import strip_chr
from .schema import ReadTable, SiteTable
from .tableio import load_tables

_npz_cache: Dict[str, tuple] = {}
_registry: Dict[str, object] = {}


def register_tables(name: str, sites: Optional[SiteTable] = None, reads: Optional[ReadTable] = None) -> None:
    """Bind an in-memory table to a file name (``--sites`` / bam path) -- used by tests and by
    callers that decode their inputs themselves."""
    _registry[name] = (sites, reads)


def is_registered(name: str) -> bool:
    """True for a name bound to in-memory tables with register_tables() (such a name needs no file)."""
    return name in _registry


def _npz(name):
    if name not in _npz_cache:
        _npz_cache[name] = load_tables(name)
    return _npz_cache[name]


def _toggle(chrom: str) -> str:
    return strip_chr(chrom) if "chr" in chrom else "chr" + chrom


def is_indexed_vcf(name: str) -> bool:
    """An existing ``*.vcf.gz`` / ``*.vcf.bgz`` file with a ``.tbi`` or ``.csi`` next to it: read natively by
    ``vcfio``."""
    return name.endswith((".vcf.gz", ".vcf.bgz")) and os.path.isfile(name) and vcfio.index_path(name) is not None


def is_indexed_bcf(name: str) -> bool:
    """An existing BGZF-compressed ``*.bcf`` file with a ``.csi`` next to it that is not a BCF of another version than
    2.2: read natively by ``bcfio`` (whose reader rejects a file that is not BCF at all)."""
    if not (name.endswith(".bcf") and os.path.isfile(name) and bcfio.index_path(name) is not None):
        return False
    with open(name, "rb") as f:
        if f.read(4) != b"\x1f\x8b\x08\x04":
            return False                               # uncompressed BCF
    head, _ = bamio.BgzfReader(name).stream_from(0, 5)
    magic = head[:5].tobytes()
    return not (magic[:3] == b"BCF" and magic != bcfio.MAGIC)


def load_sites(vcf_name: str, dnms: List[dict], pedigrees: dict, search_dist: int, engine=None) -> SiteTable:
    """The SiteTable of the trios of the DNM list around their DNMs.  An indexed ``.vcf.gz`` is read by ``vcfio`` and a
    CSI-indexed BCF 2.2 by ``bcfio`` (with ``engine``, their genotype fields are decoded on that engine's GPU); other
    BCF and unindexed files go through cyvcf2."""
    if vcf_name in _registry and _registry[vcf_name][0] is not None:
        return _registry[vcf_name][0]
    if vcf_name.endswith(".npz"):
        return _npz(vcf_name)[0]
    native = is_indexed_vcf(vcf_name)
    bcf = not native and is_indexed_bcf(vcf_name)
    if native:
        vf = vcfio.VcfFile(vcf_name)
        prefix = vf.prefix
    elif bcf:
        vf = bcfio.BcfFile(vcf_name)
        prefix = vf.prefix
    else:
        from cyvcf2 import VCF
        from .utils import get_prefix
        prefix = get_prefix(VCF(vcf_name))
    trios, seen = [], set()
    for d in dnms:
        ped = pedigrees.get(d["kid"])
        if ped and d["kid"] not in seen:
            seen.add(d["kid"])
            trios.append((d["kid"], ped["dad"], ped["mom"]))
    regions: Dict[str, List[Tuple[int, int]]] = {}
    for d in dnms:
        contig = prefix + strip_chr(d["chrom"])
        s, e = int(d["start"]), int(d["end"])
        regions.setdefault(contig, []).append((s - search_dist - 2, e + search_dist + 2))
    if native:
        return vcfio.read_sites(vf, trios, regions, engine=engine)
    if bcf:
        return bcfio.read_sites(vf, trios, regions, engine=engine)
    return packers.pack_sites(VCF(vcf_name), trios, regions)


def is_indexed_bam(name: str) -> bool:
    """An existing ``*.bam`` file with a ``.bai`` or ``.csi`` next to it: read natively by ``bamio``."""
    return name.endswith(".bam") and os.path.isfile(name) and bamio.index_path(name) is not None


def _regions(dnms, heads, has_contig, search_dist, readlen):
    regions: Dict[str, Dict[str, List[Tuple[int, int]]]] = {}
    for d in dnms:
        kid = d["kid"]
        h = heads[kid]
        cul = int(np.percentile(np.abs(h - 2 * readlen), 99.5)) if h.shape[0] else 0
        margin = max(search_dist, cul) + 2 * readlen + 2
        chrom = d["chrom"]
        if not has_contig(kid, chrom):
            chrom = _toggle(chrom)
        for p in {int(d["start"]), int(d["end"])}:
            regions.setdefault(kid, {}).setdefault(chrom, []).append((p - margin, p + margin))
    return regions


def load_reads(dnms: List[dict], search_dist: int, readlen: int, insert_size_max_sample: int, engine=None,
               min_gt_qual=20) -> Optional[ReadTable]:
    """One ReadTable for all kids of the DNM list (their ``bam`` entries name the files).

    When every file is an indexed BAM or a CRAM 3.0 with a ``.crai`` and a plain FASTA ``cram_ref`` it is read by
    ``bamio`` / ``cramio`` (no pysam; with ``engine`` the CRAM slices are decoded on the GPU too).  With ``engine`` the bases and qualities
    are then decoded on that engine's GPU: the table has no ``qual`` / ``seq2`` and carries its ``DeviceReads`` for
    the base-quality threshold of ``min_gt_qual`` (``table.device_reads``).  Every other input goes through pysam."""
    bam_of: Dict[str, str] = {}
    for d in dnms:
        bam_of.setdefault(d["kid"], d["bam"])
    if not bam_of:
        return None
    names = set(bam_of.values())
    if len(names) == 1:
        name = next(iter(names))
        if name in _registry and _registry[name][1] is not None:
            return _registry[name][1]
        if name.endswith(".npz"):
            return _npz(name)[1]
    reg = [_registry[n][1] for n in names if n in _registry and _registry[n][1] is not None]
    if reg and all(r is reg[0] for r in reg) and len(reg) == len(names):
        return reg[0]
    ref_of = {kid: next((d.get("cram_ref") for d in dnms if d["kid"] == kid), None) for kid in bam_of}
    if all(is_indexed_bam(name) or cramio.is_native_cram(name, ref_of[kid]) for kid, name in bam_of.items()):
        files = {kid: bamio.BamFile(name) if is_indexed_bam(name) else cramio.CramFile(name, ref_of[kid], engine=engine)
                 for kid, name in bam_of.items()}
        heads = {kid: f.head_tlen(insert_size_max_sample + 1) for kid, f in files.items()}
        regions = _regions(dnms, heads, lambda kid, c: c in files[kid].tids, search_dist, readlen)
        table = bamio.read_regions(files, regions, engine=engine, min_gt_qual=min_gt_qual)
        table.head_tlen = heads
        return table
    import pysam
    bams = {}
    for kid, name in bam_of.items():
        cram_ref = next((d.get("cram_ref") for d in dnms if d["kid"] == kid), None)
        bam = pysam.AlignmentFile(name, "rc", reference_filename=cram_ref) if name[-4:] == "cram" else pysam.AlignmentFile(name, "rb")
        bams[kid] = bam
    table = None
    # the insert-size estimate needs the head of every file first; then fetch around the DNMs
    heads = {}
    for kid, bam in bams.items():
        tl = []
        for i, r in enumerate(bam):
            tl.append(r.tlen)
            if i >= insert_size_max_sample:
                break
        heads[kid] = np.array(tl, dtype=np.int64)

    def has_contig(kid, chrom):
        try:
            bams[kid].fetch(chrom, 0, 1)
        except ValueError:
            return False
        return True

    regions = _regions(dnms, heads, has_contig, search_dist, readlen)
    table = packers.pack_reads(bams, regions)
    table.head_tlen = heads
    return table
