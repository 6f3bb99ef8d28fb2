"""Drop-in for the reference's ``unfazed/snv_phaser.py``: ``phase_snvs`` keeps the 20 positional
arguments of the reference (:356-377) and returns the same ``key -> record`` dict (:187-203), but
the whole DNM list is phased in one batch on the GPU (site classification, seed reads, extended
chaining, site matching, evidence tally) instead of one thread-pool task per DNM."""
from __future__ import annotations

import sys

from . import datasource
from .informative_site_finder import get_engine
from .plan import FindManyKeyError

QUIET_MODE = False


def _say(msg):
    if not QUIET_MODE:
        print(msg, file=sys.stderr)


def phase_by_reads(matches):
    """Per-variant interface of the reference (``snv_phaser.py:16-70``, repeated at ``sv_phaser.py:14-68``) for callers
    that hold ``match_informative_sites`` output: every (read, matched site) whose base at the site is the site's REF
    or ALT allele becomes an evidence item ``[read, pos]``, credited to the site's alt_parent when the read's origin
    (REF base -> ref_parent) and its haplotype relative to the DNM agree in being "ref", else to ref_parent (truth
    table :52-69).  The batched path does this in ``chain_evidence_kernel``; this is the host mirror."""
    credit = {}
    for hap, infos in matches.items():
        for info in infos:
            read = info["read"]
            for site in info["matches"]:
                if not credit:
                    credit[site["ref_parent"]] = []
                    credit[site["alt_parent"]] = []
                positions = read.get_reference_positions(full_length=True)
                if site["pos"] not in positions:
                    continue
                base = read.query_sequence[positions.index(site["pos"])]
                if base == site["ref_allele"]:
                    from_ref_parent = True
                elif base == site["alt_allele"]:
                    from_ref_parent = False
                else:
                    continue
                side = "alt_parent" if from_ref_parent == (hap == "ref") else "ref_parent"
                credit[site[side]].append([read, site["pos"]])
    return credit


def get_refalt(chrom, pos, vcf_filehandle, kid_idx):
    """``snv_phaser.py:73-84``: REF of the first record the sites VCF returns for ``chrom:pos-(pos+1)`` (contig spelled
    with the VCF's own prefix) and the ALT alleles of ALL records there, other trios' included (Q22); ``kid_idx`` is not
    used by the reference either.  The batched path takes both from the site table (``plan.SiteIndex.refalt``); this is
    the per-variant mirror for callers that hold a cyvcf2 handle."""
    from .utils import get_prefix
    region = "{}{}:{}-{}".format(get_prefix(vcf_filehandle), chrom.strip("chr"), pos, int(pos) + 1)
    ref, alts = None, []
    for record in vcf_filehandle(region):
        ref = record.REF if ref is None else ref
        alts.extend(record.ALT)
    return ref, alts


def autophase(denovo, pedigrees, records, dad_id, mom_id, build):
    """``snv_phaser.py:302-352``: a DNM of a male kid on X or Y outside the pseudoautosomal regions needs no evidence;
    its SEX-CHROM record is written into ``records`` and True is returned.  The batched path flags these entries in
    the plan (``plan.is_autophaseable``) and emits the same record (``phaser.BatchPhaser._auto_record``)."""
    from .phaser import BatchPhaser, dnm_key
    from .plan import is_autophaseable
    if not is_autophaseable(denovo, pedigrees, build):
        return False
    records[dnm_key(denovo)] = BatchPhaser._auto_record(denovo, dad_id, mom_id)
    return True


def run_batch(snvs, svs, pedigrees, sites, threads, build, no_extended, multiread_proc_min, ab_homref, ab_homalt,
              ab_het, min_gt_qual, min_depth, search_dist, insert_size_max_sample, stdevs, min_map_qual, readlen,
              split_error_margin, compact=False):
    from .phaser import BatchPhaser
    dnms = list(svs) + list(snvs)
    # an indexed sites VCF has its genotype fields decoded on the engine's GPU
    site_table = datasource.load_sites(sites, dnms, pedigrees, search_dist, engine=get_engine())
    # indexed BAM inputs are decoded on the engine's GPU; the table then comes with its device columns
    read_table = datasource.load_reads(dnms, search_dist, readlen, insert_size_max_sample, engine=get_engine(),
                                       min_gt_qual=min_gt_qual)
    bp = BatchPhaser(get_engine(), site_table, read_table, pedigrees, dreads=getattr(read_table, "device_reads", None))
    try:
        res, layout = bp.run(snvs, svs, threads=threads, build=build, no_extended=no_extended,
                             multiread_proc_min=multiread_proc_min, ab_homref=ab_homref, ab_homalt=ab_homalt,
                             ab_het=ab_het, min_gt_qual=min_gt_qual, min_depth=min_depth, search_dist=search_dist,
                             insert_size_max_sample=insert_size_max_sample, stdevs=stdevs, min_map_qual=min_map_qual,
                             readlen=readlen, split_error_margin=split_error_margin)
    except FindManyKeyError as e:
        raise KeyError(str(e))
    for name in ("sv_read", "snv"):
        for d in range(*layout[name]):
            dn = res.plan.entries[d]
            if res.plan.dnm["flags"][d] & 1 or not res.plan.found[d]:
                continue
            if res.n_cand[d] == 0:
                _say("No usable informative sites for variant {}:{}-{}".format(dn["chrom"], dn["start"], dn["end"]))
            elif res.plan.dnm["kind"][d] == 0:
                _say("No usable genotype for variant {}:{}-{}".format(dn["chrom"], dn["start"], dn["end"]))
            elif res.tally is not None and not res.tally["has_record"][d]:
                _say("No reads overlap informative sites for variant {}:{}-{}".format(dn["chrom"], dn["start"], dn["end"]))
    return bp._deliver(res, layout, compact)


def phase_snvs(dnms, kids, pedigrees, sites, threads, build, no_extended, multithread_proc_min, quiet_mode,
               ab_homref, ab_homalt, ab_het, min_gt_qual, min_depth, search_dist, insert_size_max_sample,
               stdevs, min_map_qual, readlen, split_error_margin):
    global QUIET_MODE
    QUIET_MODE = quiet_mode
    return run_batch(dnms, [], pedigrees, sites, threads, build, no_extended, multithread_proc_min, ab_homref,
                     ab_homalt, ab_het, min_gt_qual, min_depth, search_dist, insert_size_max_sample, stdevs,
                     min_map_qual, readlen, split_error_margin)


def phase_snvs_compact(dnms, kids, pedigrees, sites, threads, build, no_extended, multithread_proc_min, quiet_mode,
                       ab_homref, ab_homalt, ab_het, min_gt_qual, min_depth, search_dist, insert_size_max_sample,
                       stdevs, min_map_qual, readlen, split_error_margin):
    """``phase_snvs`` for a rank of a multi-GPU run: the same batch, returned as phaser.CompactRecords (arrays) so that
    the gather on rank 0 does not unpickle finished dicts; ``shard.merge_part`` turns it into the record dict."""
    global QUIET_MODE
    QUIET_MODE = quiet_mode
    return run_batch(dnms, [], pedigrees, sites, threads, build, no_extended, multithread_proc_min, ab_homref,
                     ab_homalt, ab_het, min_gt_qual, min_depth, search_dist, insert_size_max_sample, stdevs,
                     min_map_qual, readlen, split_error_margin, compact=True)
