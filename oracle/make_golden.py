"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/*.npz + *.json by running the UNMODIFIED
reference (the checkout named by $UNFAZED_REFERENCE, over oracle/fakes.py) on small seeded synthetic
trios and on hand-written unit vectors.  It needs no GPU:

    UNFAZED_REFERENCE=/path/to/unfazed python -m oracle.make_golden

The fixtures pin oracle/port.py (tests/test_oracle_golden.py, CPU) and the CUDA path
(tests/test_gpu_golden.py, GPU) to what the reference itself produced; reference_answers.json.gz
holds the reference's answers to the CPU tests that compare the drop-in modules and the port
with it on generated inputs.
"""
from __future__ import annotations

import copy
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import fakes, ref_driver  # noqa: E402
from unfazed_b200.synth import SynthConfig, make_dataset  # noqa: E402
from unfazed_b200.tableio import save_tables  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")

CASES = {
    "snv_noisy": (SynthConfig(dnms_per_trio=8, seed=101, coverage=24.0), {}),
    "indel_cluster_many": (SynthConfig(dnms_per_trio=8, seed=102, coverage=24.0, cluster_frac=0.4, indel_frac=0.4),
                           {"multiread_proc_min": 1}),
    "sv_cnv": (SynthConfig(dnms_per_trio=8, seed=103, coverage=24.0, sv_frac=0.75, sv_max_len=40000), {}),
    "sexchrom_chr": (SynthConfig(dnms_per_trio=8, seed=104, coverage=24.0, sex_chrom_frac=0.5, male_frac=1.0,
                                 chr_prefix="chr", sv_frac=0.25, sv_max_len=5000), {"build": "37"}),
    "no_extended": (SynthConfig(dnms_per_trio=8, seed=105, coverage=24.0), {"no_extended": True}),
}


def _norm(rec):
    r = copy.deepcopy(rec)
    for k in ("dad_sites", "mom_sites", "dad_reads", "mom_reads", "cnv_dad_sites", "cnv_mom_sites"):
        if isinstance(r[k], list):
            r[k] = sorted(r[k])
    return r


def cli_files(ds, tmp):
    """BED + PED + empty alignment files for a dataset; returns (bed, ped, bam_pairs)."""
    bed = os.path.join(tmp, "dnms.bed")
    with open(bed, "w") as f:
        f.write("#chrom\tstart\tend\tkid\tvartype\n")
        for d in ds.dnms:
            f.write("%s\t%d\t%d\t%s\t%s\n" % (d["chrom"], d["start"], d["end"], d["kid"], d["vartype"]))
    ped = os.path.join(tmp, "trio.ped")
    with open(ped, "w") as f:
        for kid, p in ds.pedigrees.items():
            f.write("fam\t%s\t%s\t%s\t%s\t2\n" % (kid, p["dad"], p["mom"], p["sex"]))
    pairs = []
    for kid in ds.pedigrees:
        path = os.path.join(tmp, kid + ".bam")
        open(path, "w").close()
        pairs.append([kid, path])
    return bed, ped, pairs


def cli_golden(ds, params):
    """BED text the reference's own ``unfazed(args)`` writes for this dataset (verbose, ambiguous
    included and excluded)."""
    import argparse
    import tempfile
    m = ref_driver.modules()
    ref_driver.register(ds)
    ref_driver.reset_state()
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        bed, ped, pairs = cli_files(ds, tmp)
        for k, (kid, path) in enumerate(pairs):
            fakes.register_bam(path, ds.reads, ds.reads.kids.index(kid))
        p = dict(ref_driver.DEFAULTS)
        p.update(params)
        for amb in (False, True):
            outfile = os.path.join(tmp, "out.bed")
            args = argparse.Namespace(
                dnms=bed, sites=ds.vcf_name, ped=ped, bam_dir=None, bam_pairs=pairs, threads=p["threads"], output_type="bed",
                include_ambiguous=amb, verbose=True, outfile=outfile, reference=None, build=p["build"],
                no_extended=p["no_extended"], multiread_proc_min=p["multiread_proc_min"], quiet=True,
                min_gt_qual=p["min_gt_qual"], min_depth=p["min_depth"], ab_homref=p["ab_homref"], ab_homalt=p["ab_homalt"],
                ab_het=p["ab_het"], evidence_min_ratio=p["evidence_min_ratio"], search_dist=p["search_dist"],
                insert_size_max_sample=p["insert_size_max_sample"], min_map_qual=p["min_map_qual"], stdevs=p["stdevs"],
                readlen=p["readlen"], split_error_margin=p["split_error_margin"], max_reads=100)
            ref_driver.reset_state()
            m["unfazed"].unfazed(args)
            out["ambiguous" if amb else "strict"] = open(outfile).read()
    return out


def dataset_cases():
    for name, (cfg, params) in CASES.items():
        ds = make_dataset(cfg)
        recs = ref_driver.phase(ds, **params)
        m = ref_driver.modules()
        ut = m["utils"]
        snvs = [d for d in ds.dnms if d["vartype"].upper() in ut.SNV_TYPES]
        svs = [d for d in ds.dnms if d["vartype"].upper() in ut.SV_TYPES]
        finds = {}
        for label, dn, wr in (("snv_read", snvs, False), ("sv_read", svs, False), ("sv_cnv", svs, True)):
            if not dn:
                continue
            try:
                ann = ref_driver.find(ds, dn, wr, **params)
                finds[label] = [{k: d.get(k) for k in ("chrom", "start", "end", "kid", "vartype", "candidate_sites", "het_sites")
                                 if k in d} for d in ann]
            except Exception as e:  # reference-undefined inputs (Q12)
                finds[label] = {"raises": type(e).__name__}
        summ = {}
        for amb in (True, False):
            s = ref_driver.summarize(copy.deepcopy(recs), include_ambiguous=amb, verbose=False)
            summ["ambiguous" if amb else "strict"] = s
        cli = cli_golden(ds, params)
        save_tables(os.path.join(OUT, name + ".npz"), ds.sites, ds.reads,
                    meta={"dnms": ds.dnms, "pedigrees": ds.pedigrees, "params": params, "truth": ds.truth})
        with open(os.path.join(OUT, name + ".json"), "w") as f:
            json.dump({"records": {k: _norm(v) for k, v in recs.items()}, "find": finds, "summary": summ, "cli": cli,
                       "generator": "oracle/make_golden.py over /root/reference (unfazed 1.0.3)"}, f, indent=0, sort_keys=True)
        print(name, "dnms", len(ds.dnms), "records", len(recs), "reads", ds.reads.n_reads)


def unit_vectors():
    """Known answers straight from the reference's own functions."""
    m = ref_driver.modules()
    isf, ss, un = m["informative_site_finder"], m["site_searcher"], m["unfazed"]
    out = {}
    # is_high_quality_site / get_kid_allele at the allele-balance boundaries (Q4, Q5)
    isf.MIN_AB_HET, isf.MAX_AB_HET = 0.2, 0.8
    isf.MIN_AB_HOMREF, isf.MAX_AB_HOMREF = 0.0, 0.2
    isf.MIN_AB_HOMALT, isf.MAX_AB_HOMALT = 0.8, 1.0
    isf.MIN_GT_QUAL, isf.MIN_DEPTH = 20, 10
    hq = []
    rng = np.random.default_rng(5)
    depth_pairs = [(12, 3), (3, 12), (67, 33), (33, 67), (10, 5), (20, 10), (30, 0), (0, 30), (5, 4), (0, 0), (-1, -1),
                   (8, 2), (2, 8), (50, 50), (1, 99), (99, 1), (4, 1), (6, 4)]
    depth_pairs += [tuple(int(x) for x in rng.integers(0, 60, size=2)) for _ in range(40)]
    for rd, ad in depth_pairs:
        for gt in (0, 1, 2, 3):
            for gq in (19.9, 20.0, 99.0):
                r = isf.is_high_quality_site(0, np.array([rd], dtype=np.int32), np.array([ad], dtype=np.int32),
                                             np.array([gt]), np.array([gq], dtype=np.float32))
                hq.append([rd, ad, gt, gq, bool(r)])
    out["is_high_quality_site"] = hq
    ka = []
    for vt in ("DEL", "DUP", "INV"):
        for _ in range(120):
            rd = rng.integers(0, 40, size=3).astype(np.int32)
            ad = rng.integers(0, 40, size=3).astype(np.int32)
            gts = rng.integers(0, 4, size=3)
            with np.errstate(all="ignore"):
                r = isf.get_kid_allele({"vartype": vt}, gts, rd, ad, 0, 1, 2)
            ka.append([vt, rd.tolist(), ad.tolist(), gts.tolist(), r])
        for rd0, ad0 in ((33, 67), (67, 33), (10, 20), (20, 10), (34, 66), (3, 3), (2, 9)):
            rd = np.array([rd0, 15, 15], dtype=np.int32)
            ad = np.array([ad0, 15, 0], dtype=np.int32)
            with np.errstate(all="ignore"):
                r = isf.get_kid_allele({"vartype": vt}, np.array([1, 1, 0]), rd, ad, 0, 1, 2)
            ka.append([vt, rd.tolist(), ad.tolist(), [1, 1, 0], r])
    out["get_kid_allele"] = ka
    # binary_search edge cases (Q16)
    bs = []
    lists = [[], [100], [100, 100], [100, 200, 300], [100, 200, 200, 300, 400], list(range(0, 5000, 137))]
    for pos in lists:
        sites = [{"pos": p} for p in pos]
        for start, end in ((0, 100), (100, 100), (100, 101), (50, 200), (150, 200), (200, 200), (199, 301), (0, 10000),
                           (300, 400), (301, 399), (401, 500), (137, 274), (138, 274), (4900, 5100)):
            bs.append([pos, start, end, [s["pos"] for s in ss.binary_search(start, end, sites)]])
    out["binary_search"] = bs
    # autophaseable at the PAR boundaries, both builds (Q6)
    ap = []
    ped = {"m": {"sex": "1"}, "f": {"sex": "2"}}
    for build in ("37", "38", "na"):
        for chrom in ("X", "chrX", "Y", "chrY", "x", "1"):
            for start in (10000, 10001, 60000, 60001, 2649520, 2649521, 2699520, 2699521, 2781479, 2781480, 5000000,
                          154931043, 154931044, 155260560, 155260561, 155701383, 156030895, 156030896, 56887903,
                          57217415, 57217416, 59034050, 59363566, 59363567):
                for kid in ("m", "f"):
                    ap.append([build, chrom, start, kid, bool(isf.autophaseable({"chrom": chrom, "start": start, "kid": kid}, ped, build))])
    out["autophaseable"] = ap
    # summarize_record decision table
    sr = []
    base = {"region": {"chrom": "1", "start": 5, "end": 6}, "vartype": "POINT", "kid": "k", "dad": "D", "mom": "M"}
    for nd in (0, 1, 2, 10, 11):
        for nm in (0, 1, 2, 10):
            for cd in (0, 1, 3, 10):
                for cm in (0, 1, 3):
                    rec = dict(base)
                    rec.update(dad_reads=["r%d" % i for i in range(nd)], mom_reads=["s%d" % i for i in range(nm)],
                               dad_sites=[str(100 + i) for i in range(min(nd, 3))], mom_sites=[str(200 + i) for i in range(min(nm, 2))],
                               cnv_dad_sites=[str(300 + i) for i in range(cd)], cnv_mom_sites=[str(400 + i) for i in range(cm)],
                               evidence_type="readbacked" if (nd or nm) else "", cnv_evidence_type="ALLELE-BALANCE" if (cd or cm) else "")
                    for amb in (True, False):
                        r = un.summarize_record(copy.deepcopy(rec), amb, True, 10)
                        sr.append([nd, nm, cd, cm, amb, r])
    out["summarize_record"] = sr
    with open(os.path.join(OUT, "unit_vectors.json"), "w") as f:
        json.dump(out, f)
    print("unit vectors:", {k: len(v) for k, v in out.items()})


def reference_answers(driver=ref_driver):
    """The answers of ``driver`` (the reference) to the tests that compare the project with it on generated inputs:
    every ``ANSWERS`` entry of the modules in ``tests.golden_util.ANSWER_MODULES``, into one gzip'd JSON file."""
    import gzip
    import importlib
    from tests import golden_util
    out = {}
    for name in golden_util.ANSWER_MODULES:
        for test, answers in importlib.import_module("tests." + name).ANSWERS.items():
            out[test] = golden_util.canon(answers(driver))
    with open(golden_util.ANSWERS_FILE, "wb") as raw, gzip.GzipFile(fileobj=raw, mode="wb", mtime=0) as f:
        f.write(json.dumps(out, sort_keys=True).encode())
    print("reference answers:", {k: len(v) for k, v in out.items()})


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    dataset_cases()
    unit_vectors()
    reference_answers()
