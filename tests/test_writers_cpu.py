"""CPU: the output writers. `write_vcf_output` and `write_bed_output` of the drop-in against the reference's
own (`unfazed/unfazed.py:336-515`, answers stored in tests/golden/reference_answers.json.gz): the VCF writer over
a recording cyvcf2 stand-in (same header additions, same phased genotypes, same UOPS / UET arrays for every variant
and sample), the BED writer's rows."""
import copy
import os
import sys
import tempfile
import types
from unittest import mock

import numpy as np
import pytest

from oracle import port
from tests.golden_util import PROJECT, assert_reference_answers
from tests.util import port_params
from unfazed_b200.synth import SynthConfig, make_dataset


class _Variant:
    def __init__(self, chrom, start, end, svtype, n_samples, het_index):
        self.CHROM, self.start, self.end = chrom, start, end
        self.INFO = {"SVTYPE": svtype} if svtype else {}
        self.genotypes = [[0, 1, False] if i == het_index else [0, 0, False] for i in range(n_samples)]
        self.gt_types = np.array([1 if i == het_index else 0 for i in range(n_samples)])
        self.formats = {}

    def set_format(self, name, arr):
        self.formats[name] = np.asarray(arr).tolist()


class _Log:
    def __init__(self):
        self.header, self.formats, self.records = [], [], []


def _cyvcf2(variants, samples, log):
    class VCF:
        def __init__(self, name):
            self.samples = list(samples)

        def add_to_header(self, line):
            log.header.append(line)

        def add_format_to_header(self, d):
            log.formats.append(dict(d))

        def __iter__(self):
            return iter(copy.deepcopy(variants))

    class Writer:
        def __init__(self, outfile, vcf):
            pass

        def write_record(self, v):
            log.records.append((v.CHROM, v.start, v.end, copy.deepcopy(v.genotypes), dict(v.formats)))

    return VCF, Writer


def _vcf_written(ref, include_ambiguous):
    """Header lines (the version written as V), FORMAT definitions and records the writer hands to cyvcf2."""
    ds = make_dataset(SynthConfig(dnms_per_trio=14, seed=401, coverage=20.0, n_trios=2, sv_frac=0.3, sv_max_len=20000,
                                  sex_chrom_frac=0.2, male_frac=1.0))
    records = port.Phaser(ds.sites, ds.reads, ds.pedigrees, port_params()).phase(copy.deepcopy(ds.dnms))
    assert len(records) >= 5
    samples = []
    for kid, ped in ds.pedigrees.items():
        samples += [kid, ped["dad"], ped["mom"]]
    variants = []
    for d in ds.dnms:
        vt = d["vartype"] if d["vartype"] in ("DEL", "DUP", "INV", "CNV", "DUP:TANDEM", "DEL:ME", "CPX", "CTX") else None
        variants.append(_Variant(d["chrom"], int(d["start"]), int(d["end"]), vt, len(samples), samples.index(d["kid"])))
    log = _Log()
    VCF, Writer = _cyvcf2(variants, samples, log)
    # the reference binds VCF and Writer at import, the drop-in imports cyvcf2 when called: both see the stand-in
    fake = types.ModuleType("cyvcf2")
    fake.VCF, fake.Writer, fake.__fake__ = VCF, Writer, True
    mod = ref.modules()["unfazed"]
    with mock.patch.object(mod, "VCF", VCF, create=True), mock.patch.object(mod, "Writer", Writer, create=True), \
            mock.patch.dict(sys.modules, {"cyvcf2": fake}):
        mod.write_vcf_output("dnms.vcf", copy.deepcopy(records), include_ambiguous, True, "out.vcf", 10)
    return {"header": [h.replace(mod.__version__, "V") for h in log.header], "formats": log.formats, "records": log.records}


def _bed_rows(ref, include_ambiguous, verbose):
    """The rows ``write_bed_output`` writes (the read-name columns are a joined Python set in the reference, Q23:
    sorted)."""
    ds = make_dataset(SynthConfig(dnms_per_trio=14, seed=402, coverage=20.0, n_trios=2, sv_frac=0.3, sv_max_len=20000,
                                  sex_chrom_frac=0.2, male_frac=1.0))
    records = port.Phaser(ds.sites, ds.reads, ds.pedigrees, port_params()).phase(copy.deepcopy(ds.dnms))
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "out.bed")
        ref.modules()["unfazed"].write_bed_output(copy.deepcopy(records), include_ambiguous, verbose, path, 10)
        out = []
        for line in open(path).read().strip().split("\n"):
            f = line.split("\t")
            if not line.startswith("#") and len(f) == 13:
                f[10] = ",".join(sorted(f[10].split(",")))
                f[12] = ",".join(sorted(f[12].split(",")))
            out.append(f)
    return out


VCF_CASES = [False, True]
BED_CASES = [(False, False), (True, True), (False, True)]
ANSWERS = {
    "test_vcf_writer_matches_reference": lambda ref: {str(a): _vcf_written(ref, a) for a in VCF_CASES},
    "test_bed_writer_matches_reference": lambda ref: {"%s-%s" % c: _bed_rows(ref, *c) for c in BED_CASES},
}


@pytest.mark.parametrize("include_ambiguous", VCF_CASES)
def test_vcf_writer_matches_reference(include_ambiguous):
    got = _vcf_written(PROJECT, include_ambiguous)
    for key in ("header", "formats", "records"):
        assert_reference_answers("test_vcf_writer_matches_reference", got[key], str(include_ambiguous), key)
    assert len(got["records"]) == 2 * 14                  # every variant is written: 2 trios x 14 DNMs
    assert sum(1 for r in got["records"] for g in r[3] if g[2] is True) >= 3


@pytest.mark.parametrize("include_ambiguous,verbose", BED_CASES)
def test_bed_writer_matches_reference(include_ambiguous, verbose):
    got = _bed_rows(PROJECT, include_ambiguous, verbose)
    assert_reference_answers("test_bed_writer_matches_reference", got, "%s-%s" % (include_ambiguous, verbose))
    assert got[0][0].startswith("#") and len(got) > 3
