"""CPU: the input readers of the orchestrator (`read_vars_bed`, `read_vars_vcf`, `get_bam_names`, `parse_ped`,
`unfazed/unfazed.py:21-160`) against the reference's answers (tests/golden/reference_answers.json.gz)."""
import contextlib
import io
import os
import sys
import tempfile
import types
from unittest import mock

import numpy as np
import pytest

from tests.golden_util import PROJECT, assert_reference_answers, reference_answer

BED = ("#chrom\tstart\tend\tkid\tvartype\n1\t100\t101\tk1\tPOINT\nchr2\t5\t900\tk2\tDEL\n"
       "X\t7\t8\tk1\tweird\n3\t10\t40\tk3\tDUP\n4\t1\t2\tk1\tINDEL\n")
PED = "f\tk1\td1\tm1\t1\t2\nf\tk2\t0\tm2\t2\t2\nf\td1\t0\t0\t1\t1\nf\tk4\td4\tm4\t2\t2\n"


def _bed_reader(ref):
    with tempfile.TemporaryDirectory() as tmp:
        bed = os.path.join(tmp, "d.bed")
        with open(bed, "w") as f:
            f.write(BED)
        return list(ref.modules()["unfazed"].read_vars_bed(bed))


def _vcf_reader(ref):
    class V:
        def __init__(self, chrom, start, end, svtype, gts):
            self.CHROM, self.start, self.end = chrom, start, end
            self.INFO = {"SVTYPE": svtype} if svtype else {}
            self.gt_types = np.array(gts)

    variants = [V("1", 10, 11, None, [1, 0, 0]), V("2", 50, 900, "DEL", [0, 3, 1]), V("X", 5, 6, None, [2, 2, 0]),
                V("3", 1, 2, "INV", [3, 3, 3])]

    class VCF:
        samples = ["a", "b", "c"]

        def __init__(self, name):
            pass

        def __iter__(self):
            return iter(variants)

    # the reference binds cyvcf2.VCF at import, the drop-in imports cyvcf2 when called: both see the stand-in
    fake = types.ModuleType("cyvcf2")
    fake.VCF, fake.__fake__ = VCF, True
    mod = ref.modules()["unfazed"]
    with mock.patch.object(mod, "VCF", VCF, create=True), mock.patch.dict(sys.modules, {"cyvcf2": fake}):
        return list(mod.read_vars_vcf("x.vcf"))


def _alignment_files(tmp):
    d = os.path.join(tmp, "bams")
    os.mkdir(d)
    for n in ("k1.bam", "k2.bam", "k3.cram", "note.txt"):
        open(os.path.join(d, n), "w").close()
    extra = os.path.join(tmp, "other.bam")
    open(extra, "w").close()
    fa = os.path.join(tmp, "ref.fa")
    with open(fa, "w") as f:
        f.write(">1\nA\n")
    return d, extra, fa


def _bam_names_and_ped(ref):
    """get_bam_names over a directory and explicit pairs (paths relative to the temporary directory, sorted), and
    parse_ped with its messages (sorted lines) in both quiet modes."""
    mod = ref.modules()["unfazed"]
    out = {"bam_names": [], "parse_ped": []}
    with tempfile.TemporaryDirectory() as tmp:
        d, extra, fa = _alignment_files(tmp)
        for args in ((d, None, fa), (d, [["k1", extra]], fa), (None, [["k9", extra]], None)):
            names = mod.get_bam_names(*args)
            out["bam_names"].append({k: sorted(os.path.relpath(p, tmp) for p in v) for k, v in names.items()})
        ped = os.path.join(tmp, "f.ped")
        with open(ped, "w") as f:
            f.write(PED)
        for quiet in (True, False):
            mod.QUIET_MODE = quiet
            err = io.StringIO()
            with contextlib.redirect_stderr(err):
                entries = mod.parse_ped(ped, {"k1", "k2", "k3"})
            out["parse_ped"].append([entries, sorted(err.getvalue().splitlines())])
        mod.QUIET_MODE = False
    return out


ANSWERS = {"test_bed_reader": _bed_reader, "test_vcf_reader": _vcf_reader, "test_bam_names_and_ped": _bam_names_and_ped}


def test_bed_reader(tmp_path):
    assert_reference_answers("test_bed_reader", _bed_reader(PROJECT))
    bad = tmp_path / "bad.bed"
    bad.write_text("1\t100\t101\tk1\n")
    with pytest.raises(SystemExit) as e:
        list(PROJECT.modules()["unfazed"].read_vars_bed(str(bad)))
    assert "must contain the following columns exactly" in str(e.value)


def test_vcf_reader():
    assert_reference_answers("test_vcf_reader", _vcf_reader(PROJECT))
    assert len(reference_answer("test_vcf_reader")) == 6


def test_bam_names_and_ped(tmp_path):
    got = _bam_names_and_ped(PROJECT)
    for key in ("bam_names", "parse_ped"):
        assert_reference_answers("test_bam_names_and_ped", got[key], key)
    assert all(entries == {"k1": {"kid": "k1", "dad": "d1", "mom": "m1", "sex": "1"}} for entries, _err in got["parse_ped"])
    new = PROJECT.modules()["unfazed"]
    d, _extra, _fa = _alignment_files(str(tmp_path))
    with pytest.raises(SystemExit) as e:
        new.get_bam_names(d, None, None)
    assert str(e.value) == "Missing reference file for CRAM"
    with pytest.raises(SystemExit) as e:
        new.get_bam_names(d, None, str(tmp_path / "nope.fa"))
    assert str(e.value) == "Reference file is not valid"
    with pytest.raises(SystemExit) as e:
        new.get_bam_names(None, [["k1", str(tmp_path / "missing.bam")]], None)
    assert str(e.value).startswith("invalid filename")
