"""CPU: the command line's error paths, asserted like the reference's own functional tests
(test/func/unfazed_snv_test.sh:353-402) -- these exit before any GPU work -- plus the UET coding of
the VCF writer (unfazed.py:415-433) and the BED column layout."""
import io
import os
import sys

import pytest

from unfazed_b200 import __main__ as cli
from unfazed_b200 import unfazed as orch


def _write(tmp_path, name, text):
    p = tmp_path / name
    p.write_text(text)
    return str(p)


def _run(argv, capsys):
    with pytest.raises(SystemExit) as ei:
        cli.main(argv)
    err = capsys.readouterr().err
    msg = ei.value.code if isinstance(ei.value.code, str) else ""
    return err + "\n" + msg


@pytest.fixture
def inputs(tmp_path):
    bed = _write(tmp_path, "dnms.bed", "#chrom\tstart\tend\tkid\tvartype\n22\t18844941\t18844942\tNA12878\tPOINT\n")
    ped = _write(tmp_path, "trio.ped", "fam\tNA12878\tNA12891\tNA12892\t2\t2\nfam\tNA12891\t0\t0\t1\t1\nfam\tNA12892\t0\t0\t2\t1\n")
    bam = _write(tmp_path, "NA12878.bam", "")
    return bed, ped, bam


def test_missing_kid_from_ped(inputs, tmp_path, capsys):
    bed, _ped, bam = inputs
    ped = _write(tmp_path, "missing_kid.ped", "fam\tNA12891\t0\t0\t1\t1\nfam\tNA12892\t0\t0\t2\t1\n")
    out = _run(["-d", bed, "-s", "sites.vcf.gz", "-p", ped, "-o", "bed", "--build", "38", "--bam-pairs", "NA12878:" + bam], capsys)
    assert "NA12878 missing from pedigree file, will be skipped" in out
    assert "No phaseable variants" in out


def test_missing_dad_from_ped(inputs, tmp_path, capsys):
    bed, _ped, bam = inputs
    ped = _write(tmp_path, "missing_dad.ped", "fam\tNA12878\t0\tNA12892\t2\t2\nfam\tNA12892\t0\t0\t2\t1\n")
    out = _run(["-d", bed, "-s", "sites.vcf.gz", "-p", ped, "-o", "bed", "--build", "38", "--bam-pairs", "NA12878:" + bam], capsys)
    assert "Parent of sample NA12878 missing from pedigree file, will be skipped" in out
    assert "No phaseable variants" in out


def test_invalid_output_to_vcf(inputs, capsys):
    bed, ped, bam = inputs
    out = _run(["-d", bed, "-s", "sites.vcf.gz", "-p", ped, "-o", "vcf", "--build", "38", "--bam-pairs", "NA12878:" + bam], capsys)
    assert ("Invalid option: --output-type is vcf, but input is not a vcf type. Rerun with `--output-type bed` or input "
            "dnms as one of the following: vcf, vcf.gz, bcf") in out


def test_invalid_bam(inputs, capsys):
    bed, ped, _bam = inputs
    out = _run(["-d", bed, "-s", "sites.vcf.gz", "-p", ped, "-o", "vcf", "--build", "38", "--bam-pairs", "NA12878:bob"], capsys)
    assert "invalid filename bob" in out


def test_missing_bam_arguments(inputs, capsys):
    bed, ped, _bam = inputs
    with pytest.raises(SystemExit):
        cli.main(["-d", bed, "-s", "s.vcf.gz", "-p", ped, "--build", "38"])
    assert "Missing required argument: --bam-dir or --bam-pairs must be set" in capsys.readouterr().err


def test_flag_defaults_match_the_reference():
    a = cli.setup_args().parse_args(["-d", "x.bed", "-s", "s", "-p", "p", "-g", "38", "--bam-pairs", "k:b"])
    assert (a.threads, a.multiread_proc_min, a.min_gt_qual, a.min_depth, a.search_dist) == (2, 1000, 20, 10, 5000)
    assert (a.insert_size_max_sample, a.min_map_qual, a.stdevs, a.readlen, a.split_error_margin, a.max_reads) == (1000000, 1, 3, 151, 5, 100)
    # argparse runs string defaults through `type`, exactly as in the reference (__main__.py:157-183)
    assert a.ab_homref == [0.0, 0.2] and a.ab_het == [0.2, 0.8] and a.ab_homalt == [0.8, 1.0]
    assert a.evidence_min_ratio == 10
    b = cli.setup_args().parse_args(["-d", "x.bed", "-s", "s", "-p", "p", "-g", "37", "--bam-pairs", "k:b", "--ab-het", "0.25:0.75"])
    assert b.ab_het == [0.25, 0.75] and b.bam_pairs == [["k", "b"]]


def test_uet_codes():
    assert orch.uet_code(["READBACKED"]) == 0 and orch.uet_code(["ALLELE-BALANCE"]) == 1
    assert orch.uet_code(["READBACKED", "ALLELE-BALANCE"]) == 2 and orch.uet_code(["AMBIGUOUS_READBACKED"]) == 3
    assert orch.uet_code(["AMBIGUOUS_ALLELE-BALANCE"]) == 4 and orch.uet_code(["AMBIGUOUS_BOTH"]) == 5
    assert orch.uet_code(["SEX-CHROM"]) == 6 and orch.uet_code([]) == -1


def test_bed_writer_columns_and_order(tmp_path):
    recs = {}
    for i, (chrom, start) in enumerate([("22", 30), ("22", 10), ("3", 5)]):
        recs["k%d" % i] = {"region": {"chrom": chrom, "start": start, "end": start + 1}, "vartype": "POINT", "kid": "kid",
                           "dad": "D", "mom": "M", "dad_sites": ["7", "100"], "mom_sites": [], "evidence_type": "readbacked",
                           "dad_reads": ["r2", "r1"], "mom_reads": [], "cnv_dad_sites": "", "cnv_mom_sites": "", "cnv_evidence_type": ""}
    out = tmp_path / "o.bed"
    orch.write_bed_output(recs, False, True, str(out), 10)
    lines = out.read_text().strip().split("\n")
    assert lines[0] == ("#chrom\tstart\tend\tvartype\tkid\torigin_parent\tother_parent\tevidence_count\tevidence_types\t"
                        "origin_parent_sites\torigin_parent_reads\tother_parent_sites\tother_parent_reads")
    assert [l.split("\t")[:2] for l in lines[1:]] == [["22", "10"], ["22", "30"], ["3", "5"]]     # sorted by (chrom, start, end)
    assert lines[1].split("\t")[5:] == ["D", "M", "2", "READBACKED", "100,7", "r2,r1", "-", "-"]    # sites sorted as strings (Q23)
