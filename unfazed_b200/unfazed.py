"""Orchestrator: DNM readers, alignment-file discovery, pedigree parsing, the final evidence call
and the BED / VCF writers -- the same behaviour, flags and messages as the reference's
``unfazed/unfazed.py`` (readers :18-90, get_bam_names :93-126, parse_ped :129-159,
summarize_record :190-334, writers :337-515, unfazed :518-667).  Host-side formatting only; the
phasing itself is ``snv_phaser.phase_snvs`` / ``sv_phaser.phase_svs``."""
from __future__ import annotations

import glob
import gzip
import os
import sys

from . import __version__, datasource
from .snv_phaser import phase_snvs
from .sv_phaser import phase_svs
from .utils import HET, HOM_ALT, LABELS, SNV_TYPES, SV_TYPES, VCF_TYPES

QUIET_MODE = False
BED_MSG = "dnms bed file must contain the following columns exactly: " + ", ".join(LABELS)


def _bed_rows(handle):
    for line in handle:
        if line.startswith("#"):
            continue
        f = line.strip().split()
        if len(f) != 5:
            sys.exit(BED_MSG)
        yield {"chrom": f[0], "start": int(f[1]), "end": int(f[2]), "kid": f[3],
               "vartype": f[4] if f[4] in SV_TYPES else SNV_TYPES[0], "bam": ""}


def read_vars_bed(bedname):
    with open(bedname, "r") as fh:
        yield from _bed_rows(fh)


def read_vars_bedzip(bedzipname):
    # the reference opens the gzip in binary mode and never matches a str under Python 3 (Q25);
    # here the file is read as text so .bed.gz input actually works
    with gzip.open(bedzipname, "rt") as fh:
        yield from _bed_rows(fh)


def read_vars_vcf(vcfname):
    if os.path.isfile(vcfname):
        # an existing .vcf / .vcf.gz / .bcf: read natively (vcfio, bcfio), no cyvcf2 needed
        if vcfname.endswith(".bcf"):
            from .bcfio import read_dnms
        else:
            from .vcfio import read_dnms
        yield from read_dnms(vcfname)
        return
    from cyvcf2 import VCF
    vcf = VCF(vcfname)
    for v in vcf:
        vartype = v.INFO.get("SVTYPE") or SNV_TYPES[0]
        for i, gt in enumerate(v.gt_types):
            if gt in (HET, HOM_ALT):
                yield {"chrom": v.CHROM, "start": v.start, "end": v.end, "kid": vcf.samples[i],
                       "vartype": vartype, "bam": ""}


def get_bam_names(bam_dir, bam_pairs, cram_ref):
    found = {}
    cram = False
    if bam_dir is not None:
        for ext in ("bam", "cram"):
            for path in glob.glob(os.path.join(bam_dir, "*." + ext)):
                cram |= ext == "cram"
                found.setdefault(os.path.splitext(os.path.basename(path))[0], set()).add(path)
    for sample, path in (bam_pairs or []):
        if not os.path.isfile(path) and not datasource.is_registered(path):      # tables bound with register_tables()
            sys.exit("invalid filename " + path)
        found[sample] = {path}
        cram |= path.endswith("cram")
    if cram:
        if cram_ref is None:
            sys.exit("Missing reference file for CRAM")
        if not os.path.isfile(cram_ref):
            sys.exit("Reference file is not valid")
    return found


def parse_ped(ped, kids):
    entries, no_parents = {}, []
    with open(ped, "r") as fh:
        for line in fh:
            f = line.strip().split()
            if len(f) < 5 or f[1] not in kids:
                continue
            if f[2] == "0" or f[3] == "0":
                if not QUIET_MODE:
                    print("Parent of sample {} missing from pedigree file, will be skipped".format(f[1]), file=sys.stderr)
                no_parents.append(f[1])
                continue
            entries[f[1]] = dict(zip(["kid", "dad", "mom", "sex"], f[1:5]))
    for s in kids:
        if s not in entries and s not in no_parents and not QUIET_MODE:
            print("{} missing from pedigree file, will be skipped".format(s), file=sys.stderr)
    return entries


def summarize_record(read_record, include_ambiguous, verbose, evidence_min_ratio):
    """Final call from the per-parent evidence (reference :162-334; the same decision table runs on
    the device in unfz_summarize for the batch API)."""
    rec = read_record
    region = rec["region"]
    head = {"chrom": region["chrom"], "start": int(region["start"]), "end": int(region["end"]),
            "vartype": rec["vartype"], "kid": rec["kid"]}
    if rec["evidence_type"] == "SEX-CHROM":
        on_y = region["chrom"].lower().strip("chr") == "y"
        out = dict(head, origin_parent=rec["dad"] if on_y else rec["mom"], other_parent=rec["mom"] if on_y else rec["dad"],
                   evidence_count=1, evidence_types=["SEX-CHROM"])
        if verbose:
            out.update(origin_parent_sites="NA", origin_parent_reads="NA", other_parent_sites="NA", other_parent_reads="NA")
        return out
    r = evidence_min_ratio
    sides = {"dad": (rec["dad"], rec["dad_sites"], rec["dad_reads"], rec["cnv_dad_sites"]),
             "mom": (rec["mom"], rec["mom_sites"], rec["mom_reads"], rec["cnv_mom_sites"])}
    n = {k: len(v[2]) for k, v in sides.items()}
    c = {k: len(v[3]) for k, v in sides.items()}
    origin = other = None
    o_sites, o_reads, x_sites, x_reads, types = [], [], [], [], []
    count, ambig = 0, False

    def take(win, lose):
        nonlocal o_sites, o_reads, x_sites, x_reads
        o_sites += sides[win][1]; o_reads += sides[win][2]
        x_sites += sides[lose][1]; x_reads += sides[lose][2]

    for win, lose in (("dad", "mom"), ("mom", "dad")):
        if n[win] > 0 and n[win] >= r * n[lose]:
            origin, other, count = sides[win][0], sides[lose][0], len(sides[win][1])
            take(win, lose)
            types.append("READBACKED")
            break
    else:
        if n["dad"] > 0 and n["mom"] > 0:
            origin, count, ambig = rec["dad"] + "|" + rec["mom"], n["dad"] + n["mom"], True
            take("dad", "mom")
            types.append("AMBIGUOUS_READBACKED")
    decided = None
    for win, lose in (("dad", "mom"), ("mom", "dad")):
        if c[win] > 0 and c[win] >= r * c[lose]:
            decided = (win, lose)
            break
    if decided:
        win, lose = decided
        if origin == sides[lose][0] and "READBACKED" not in types:
            origin, ambig = None, True
            count += c["dad"] + c["mom"]
            o_sites += rec["cnv_dad_sites"]
            if win == "dad":
                x_sites = rec["cnv_mom_sites"]
            else:
                x_sites += rec["cnv_mom_sites"]
            types = ["AMBIGUOUS_BOTH"]
        else:
            origin, other, count = sides[win][0], sides[lose][0], c[win]
            o_sites += sides[win][3]; o_reads += sides[win][2]
            x_sites += sides[lose][1]; x_reads += sides[lose][2]
            if "AMBIGUOUS_READBACKED" in types:
                types.remove("AMBIGUOUS_READBACKED")
                if win == "dad":
                    ambig = False
            types.append("ALLELE-BALANCE")
    elif (c["dad"] + c["mom"]) > 0 and "READBACKED" not in types:
        origin, ambig = None, True
        count += c["dad"] + c["mom"]
        o_sites += rec["cnv_dad_sites"]
        x_sites = rec["cnv_mom_sites"]
        types.append("AMBIGUOUS_ALLELE-BALANCE")
    if (origin is None or ambig) and not include_ambiguous:
        return None
    out = dict(head, origin_parent=origin, other_parent=other, evidence_count=count, evidence_types=types)
    if verbose:
        join = lambda xs: ",".join(xs) if len(xs) > 0 else "-"
        out.update(origin_parent_sites=join(sorted(o_sites)), origin_parent_reads=join(o_reads),
                   other_parent_sites=join(sorted(x_sites)), other_parent_reads=join(x_reads))
    return out


BED_COLUMNS = ["chrom", "start", "end", "vartype", "kid", "origin_parent", "other_parent", "evidence_count", "evidence_types"]
VERBOSE_COLUMNS = ["origin_parent_sites", "origin_parent_reads", "other_parent_sites", "other_parent_reads"]


def write_bed_output(read_records, include_ambiguous, verbose, outfile, evidence_min_ratio):
    cols = BED_COLUMNS + (VERBOSE_COLUMNS if verbose else [])
    rows = [s for s in (summarize_record(rec, include_ambiguous, verbose, evidence_min_ratio)
                        for rec in read_records.values()) if s is not None]
    rows.sort(key=lambda x: (x["chrom"], x["start"], x["end"]))
    out = sys.stdout if outfile == "/dev/stdout" else open(outfile, "w")
    try:
        print("#" + "\t".join(cols), file=out)
        for row in rows:
            row = dict(row, evidence_types=",".join(row["evidence_types"]))
            print("\t".join(str(row[c]) for c in cols), file=out)
    finally:
        if out is not sys.stdout:
            out.close()


UET_CODES = [("AMBIGUOUS_READBACKED", 3), ("AMBIGUOUS_ALLELE-BALANCE", 4), ("AMBIGUOUS_BOTH", 5), ("SEX-CHROM", 6)]


def uet_code(evidence_types):
    """UET FORMAT value (reference :415-433)."""
    for name, code in UET_CODES:
        if name in evidence_types:
            return code
    rb, ab = "READBACKED" in evidence_types, "ALLELE-BALANCE" in evidence_types
    return 2 if (rb and ab) else 0 if rb else 1 if ab else -1


def write_vcf_output(in_vcf_name, read_records, include_ambiguous, verbose, outfile, evidence_min_ratio, engine=None):
    if os.path.isfile(in_vcf_name) and in_vcf_name.endswith((".vcf", ".vcf.gz")) and not outfile.endswith(".bcf"):
        # an existing text VCF written as text or BGZF: natively (vcfio), no cyvcf2 needed
        from .vcfio import write_phased_vcf
        write_phased_vcf(in_vcf_name, read_records, include_ambiguous, verbose, outfile, evidence_min_ratio, engine)
        return
    if os.path.isfile(in_vcf_name) and in_vcf_name.endswith(".bcf") and not outfile.endswith(".bcf"):
        from . import bcfio
        if bcfio.is_bcf(in_vcf_name):
            # an existing BCF 2.2 written as text or BGZF: natively (bcfio), no cyvcf2 needed
            bcfio.write_phased_vcf(in_vcf_name, read_records, include_ambiguous, verbose, outfile, evidence_min_ratio,
                                   engine)
            return
    import numpy as np
    from cyvcf2 import VCF, Writer
    vcf = VCF(in_vcf_name)
    vcf.add_to_header("##unfazed=" + __version__ + ". Phase info in pipe-separated GT field order -> 1|0 is paternal, 0|1 is maternal")
    vcf.add_format_to_header({"ID": "UOPS", "Description": "Count of pieces of evidence supporting the unfazed-identified origin parent or `-1` if missing", "Type": "Float", "Number": "1"})
    vcf.add_format_to_header({"ID": "UET", "Description": "Unfazed evidence type: `0` (readbacked), `1` (allele-balance, for CNVs only), `2` (both), `3` (ambiguous readbacked), `4` (ambiguous allele-balance), `5` (ambiguous both), `6` (auto-phased sex-chromosome variant in male), or `-1` (missing)", "Type": "Float", "Number": "1"})
    writer = Writer(outfile, vcf)
    for v in vcf:
        gts = v.genotypes
        uops, uet = [], []
        for i, gt in enumerate(v.gt_types):
            a, b = -1, -1
            if gt in (HET, HOM_ALT):
                key = "{}_{}_{}_{}_{}".format(v.CHROM, v.start, v.end, vcf.samples[i], v.INFO.get("SVTYPE") or SNV_TYPES[0])
                if key in read_records:
                    s = summarize_record(read_records[key], include_ambiguous, verbose, evidence_min_ratio)
                    if s is not None:
                        if s["origin_parent"] == read_records[key]["dad"]:
                            gts[i][0], gts[i][1], gts[i][2] = 1, 0, True
                        elif s["origin_parent"] == read_records[key]["mom"]:
                            gts[i][0], gts[i][1], gts[i][2] = 0, 1, True
                        a, b = s["evidence_count"], uet_code(s["evidence_types"])
            uops.append(a)
            uet.append(b)
        v.genotypes = gts
        v.set_format("UOPS", np.array(uops))
        v.set_format("UET", np.array(uet))
        writer.write_record(v)


def _phase_multi_gpu(snvs, svs, common):
    """One process per GPU (torchrun): DNMs shard by kid, every rank phases its shard on its own
    device and rank 0 gathers the records -- no collective on the data path.  The choice between
    ``find`` and ``find_many`` depends on the number of DNMs of the WHOLE run
    (informative_site_finder.py:190), so it is taken here and handed to the ranks as an effective
    ``multiread_proc_min`` of 0 or "never"."""
    import torch
    import torch.distributed as dist
    from . import informative_site_finder as isf
    from .shard import cross_kid_coupling, phase_sharded
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if not dist.is_initialized():
        dist.init_process_group("cpu:gloo,cuda:nccl")
    from .engine import Engine
    isf._engine = Engine(local_rank)
    pedigrees, build, mpm = common[1], common[4], common[6]

    def with_mpm(n_total):
        c = list(common)
        c[6] = 0 if n_total >= mpm else 2 ** 31 - 1
        return c

    def phase_fn(mine):
        my_svs = [d for d in mine if d["vartype"].upper() in SV_TYPES]
        my_snvs = [d for d in mine if d["vartype"].upper() in SNV_TYPES]
        if my_snvs and not my_svs:
            # the shard travels to rank 0 as arrays and becomes record dicts there (shard.merge_part)
            from .snv_phaser import phase_snvs_compact
            return phase_snvs_compact(my_snvs, *with_mpm(len(snvs)))
        out = phase_snvs(my_snvs, *with_mpm(len(snvs))) if my_snvs else {}
        out.update(phase_svs(my_svs, *with_mpm(len(svs))) if my_svs else {})
        return out

    if cross_kid_coupling(svs, pedigrees, build, mpm):
        # one kid's events change another kid's windows (Q12): the run stays on rank 0 to be exact.  It still goes
        # through the gather protocol of phase_sharded (every rank reaches the collective, an exception on rank 0
        # is re-raised after it), so a failure cannot leave the other ranks waiting
        return phase_sharded(phase_fn, svs + snvs, split_heavy=False, all_on_rank0=True)
    # a family is only cut into slices when its DNMs cannot interact (per-DNM `find` windows)
    return phase_sharded(phase_fn, svs + snvs, split_heavy=len(snvs) < mpm and len(svs) < mpm)


def unfazed(args):
    global QUIET_MODE
    QUIET_MODE = args.quiet
    bams = get_bam_names(args.bam_dir, args.bam_pairs, args.reference)
    if args.dnms.endswith(".bed"):
        reader, input_type = read_vars_bed, "bed"
    elif args.dnms.endswith(".bed.gz"):
        reader, input_type = read_vars_bedzip, "bed"
    elif any(args.dnms.endswith(t) for t in VCF_TYPES):
        reader, input_type = read_vars_vcf, "vcf"
    else:
        sys.exit("dnms file type is unrecognized. Must be bed, bed.gz, vcf, vcf.gz, or bcf")
    output_type = args.output_type if args.output_type is not None else input_type
    if output_type == "vcf" and input_type != "vcf":
        print("Invalid option: --output-type is vcf, but input is not a vcf type. "
              + "Rerun with `--output-type bed` or input dnms as one of the following:", ", ".join(VCF_TYPES), file=sys.stderr)
        sys.exit(1)
    kids, snvs, svs = set(), [], []
    warned = set()
    for var in reader(args.dnms):
        s = var["kid"]
        if s not in bams or len(bams[s]) != 1:
            if s not in warned and not QUIET_MODE:
                if s not in bams:
                    print("missing alignment file for", s, file=sys.stderr)
                else:
                    print("multiple alignment files for", s + ".", "Please specify correct alignment file using --bam-pairs", file=sys.stderr)
            warned.add(s)
            continue
        kids.add(s)
        var["bam"] = next(iter(bams[s]))
        var["cram_ref"] = args.reference
        if var["vartype"].upper() in SV_TYPES:
            svs.append(var)
        elif var["vartype"].upper() in SNV_TYPES:
            snvs.append(var)
    pedigrees = parse_ped(args.ped, kids)
    kid_list = list(pedigrees)
    snvs = [v for v in snvs if v["kid"] in pedigrees]
    svs = [v for v in svs if v["kid"] in pedigrees]
    if not snvs and not svs:
        sys.exit("No phaseable variants")
    common = (kid_list, pedigrees, args.sites, args.threads, args.build, args.no_extended, args.multiread_proc_min,
              args.quiet, args.ab_homref, args.ab_homalt, args.ab_het, args.min_gt_qual, args.min_depth,
              args.search_dist, args.insert_size_max_sample, args.stdevs, args.min_map_qual, args.readlen,
              args.split_error_margin)
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        phased = _phase_multi_gpu(snvs, svs, common)
        if phased is None:
            return                                  # ranks > 0 hold no output
    else:
        phased_svs = phase_svs(svs, *common) if svs else {}
        phased = phase_snvs(snvs, *common) if snvs else {}
        phased.update(phased_svs)
    if output_type == "vcf":
        from . import informative_site_finder
        write_vcf_output(args.dnms, phased, args.include_ambiguous, args.verbose, args.outfile, args.evidence_min_ratio,
                         informative_site_finder._engine)
    else:
        write_bed_output(phased, args.include_ambiguous, args.verbose, args.outfile, args.evidence_min_ratio)
