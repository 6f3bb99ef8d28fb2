"""CPU: the phased VCF writer without cyvcf2 (vcfio.write_phased_vcf, csrc/vcfout.cu host entry points).  The records
and header additions equal the reference's (stored answers of test_writers_cpu); hand-written lines check the output
contract byte for byte; malformed input raises; the containers and the routing of unfazed.write_vcf_output."""
import copy
import gzip
import os
import sys
from unittest import mock

import numpy as np
import pytest

from oracle import port
from tests.golden_util import reference_answer
from tests.util import port_params
from unfazed_b200 import _lib as L
from unfazed_b200 import bamio, unfazed, vcfio
from unfazed_b200.synth import SynthConfig, make_dataset

SV_TYPES = ("DEL", "DUP", "INV", "CNV", "DUP:TANDEM", "DEL:ME", "CPX", "CTX")
HEAD = "##fileformat=VCFv4.2\n"


def _cols(samples):
    return "\t".join(["#CHROM", "POS", "ID", "REF", "ALT", "QUAL", "FILTER", "INFO", "FORMAT"] + list(samples)) + "\n"


def parity_dataset(tmp_path):
    """The dataset of test_writers_cpu._vcf_written as a real .vcf.gz: (path, records, samples)."""
    ds = make_dataset(SynthConfig(dnms_per_trio=14, seed=401, coverage=20.0, n_trios=2, sv_frac=0.3, sv_max_len=20000,
                                  sex_chrom_frac=0.2, male_frac=1.0))
    records = port.Phaser(ds.sites, ds.reads, ds.pedigrees, port_params()).phase(copy.deepcopy(ds.dnms))
    samples = []
    for kid, ped in ds.pedigrees.items():
        samples += [kid, ped["dad"], ped["mom"]]
    lines = []
    for d in ds.dnms:
        s, e = int(d["start"]), int(d["end"])
        sv = d["vartype"] in SV_TYPES
        gts = ["0/1" if x == d["kid"] else "0/0" for x in samples]
        lines.append("\t".join([d["chrom"], str(s + 1), ".", "N" if sv else "N" * (e - s), "<%s>" % d["vartype"] if sv
                                else "A", ".", ".", "SVTYPE=%s;END=%d" % (d["vartype"], e) if sv else ".", "GT"] + gts))
    path = str(tmp_path / "dnms.vcf.gz")
    bamio.write_bgzf(path, (HEAD + _cols(samples)).encode(), ("\n".join(lines) + "\n").encode())
    return path, records, samples


def parse_output(text: str):
    """(header lines, records as test_writers_cpu stores them: CHROM, pos0, end, [a, b, phased] per sample, UOPS/UET)."""
    head, recs = [], []
    for line in text.rstrip("\n").split("\n"):
        if line.startswith("#"):
            head.append(line)
            continue
        f = line.split("\t")
        pos0 = int(f[1]) - 1
        info = dict(kv.partition("=")[::2] for kv in f[7].split(";"))
        end = int(info["END"]) if "END" in info else pos0 + len(f[3])
        keys = f[8].split(":")
        gts, vals = [], {"UOPS": [], "UET": []}
        for cell in f[9:]:
            sub = dict(zip(keys, cell.split(":")))
            gt = sub["GT"]
            al = [int(a) for a in gt.replace("|", "/").split("/")]
            gts.append([al[0], al[1], "|" in gt])
            for k in vals:
                vals[k].append(int(sub[k]))
        recs.append([f[0], pos0, end, gts, vals])
    return head, recs


@pytest.mark.parametrize("include_ambiguous", [False, True])
def test_parity_with_reference(tmp_path, include_ambiguous):
    path, records, _ = parity_dataset(tmp_path)
    out = str(tmp_path / "out.vcf")
    vcfio.write_phased_vcf(path, copy.deepcopy(records), include_ambiguous, True, out, 10)
    head, recs = parse_output(open(out).read())
    want = reference_answer("test_vcf_writer_matches_reference")[str(include_ambiguous)]
    assert recs == want["records"]
    assert sum(1 for r in recs for g in r[3] if g[2]) >= 3
    added = [h.replace(unfazed.__version__, "V") for h in head if h.startswith("##unfazed=")]
    assert added == want["header"]
    fmts = []
    for h in head:
        if h.startswith("##FORMAT=<ID=U"):
            body = h[len("##FORMAT=<"):-1]
            d = {}
            for part in ("ID", "Number", "Type"):
                k, _, rest = body.partition(",")
                d[part] = k.split("=", 1)[1]
                body = rest
            assert body.startswith('Description="') and body.endswith('"')
            d["Description"] = body[len('Description="'):-1]
            fmts.append(d)
    assert fmts == want["formats"]
    # the three lines sit right before #CHROM, PASS after ##fileformat
    assert head[1] == vcfio.PASS_LINE and head[-1].startswith("#CHROM") and head[-4].startswith("##unfazed=")


# ------------------------------------------------------------------------------------------------
# hand-written lines through the edit list
# ------------------------------------------------------------------------------------------------

def rewrite(lines, n_samples, edits=None, dec=None):
    """Body ``lines`` rewritten with ``edits`` {line: [(sample, phase, uops, uet)]}: (output lines, line status)."""
    text = "".join(l + "\n" for l in lines).encode()
    buf = np.frombuffer(text, dtype=np.uint8)
    dec = dec or vcfio.HostDecoder()
    recs = dec.lines(buf)
    rows = sorted((i, *e) for i, es in (edits or {}).items() for e in es)
    ed = np.zeros(len(rows), dtype=L.VCF_EDIT_DTYPE)
    for k, name in enumerate(("sample", "phase", "uops", "uet")):
        ed[name] = [r[k + 1] for r in rows]
    off = np.searchsorted(np.array([r[0] for r in rows], dtype=np.int64), np.arange(len(lines) + 1)).astype(np.int64)
    out, bad = dec.rewrite(off, ed, n_samples)
    return out.tobytes().decode().split("\n")[:-1], bad


def test_untouched_cells_byte_for_byte():
    line = "chr1\t1001\trs1\tACG\tA,AT\t50.00\tq10;LowQual\tDP=30;AF=0.5,0.1\tGT:GQ:AD:PL\t0/2:35:1,2,3:0,10,100\t./.:.:.:."
    out, bad = rewrite([line], 2)
    assert not bad.any()
    assert out == ["chr1\t1001\trs1\tACG\tA,AT\t50.00\tq10;LowQual\tDP=30;AF=0.5,0.1\tGT:GQ:AD:PL:UOPS:UET"
                   "\t0/2:35:1,2,3:0,10,100:-1:-1\t./.:.:.:.:-1:-1"]


def test_phase_dad_mom_gt_not_first_and_triploid():
    lines = ["1\t10\t.\tA\tC\t.\t.\t.\tGQ:GT:DP\t30:0/1:7\t20:1|1:8\t10:0/1/1:9"]
    out, _ = rewrite(lines, 3, {0: [(0, 1, 4, 0), (1, 2, 2, 1), (2, 1, 12345, 2)]})
    assert out == ["1\t10\t.\tA\tC\t.\t.\t.\tGQ:GT:DP:UOPS:UET\t30:1|0:7:4:0\t20:0|1:8:2:1\t10:1|0|1:9:12345:2"]


def test_ambiguous_keeps_gt_and_sets_values():
    out, _ = rewrite(["1\t10\t.\tA\tC\t.\t.\t.\tGT\t0/1\t0/0"], 2, {0: [(0, 0, 5, 3)]})
    assert out == ["1\t10\t.\tA\tC\t.\t.\t.\tGT:UOPS:UET\t0/1:5:3\t0/0:-1:-1"]


def test_dropped_subfields_and_absent_columns():
    out, _ = rewrite(["1\t10\t.\tA\tC\t.\t.\t.\tGT:GQ:AD\t0/1\t0/0:3"], 4, {0: [(0, 2, 1, 0)]})
    assert out == ["1\t10\t.\tA\tC\t.\t.\t.\tGT:GQ:AD:UOPS:UET\t0|1:.:.:1:0\t0/0:3:.:-1:-1\t.:.:.:-1:-1\t.:.:.:-1:-1"]
    # a FORMAT column without any sample column
    out, _ = rewrite(["1\t10\t.\tA\tC\t.\t.\t.\tGT"], 2)
    assert out == ["1\t10\t.\tA\tC\t.\t.\t.\tGT:UOPS:UET\t.:-1:-1\t.:-1:-1"]


def test_existing_uops_uet_replaced_in_place():
    lines = ["1\t10\t.\tA\tC\t.\t.\t.\tGT:UOPS:GQ:UET\t1|0:7:30:0\t0/0:-1:20:-1", "1\t11\t.\tA\tC\t.\t.\t.\tGT:UET\t0/1\t0/1"]
    out, _ = rewrite(lines, 2, {0: [(0, 2, 9, 1)], 1: [(1, 1, 3, 0)]})
    assert out == ["1\t10\t.\tA\tC\t.\t.\t.\tGT:UOPS:GQ:UET\t0|1:9:30:1\t0/0:-1:20:-1",
                   "1\t11\t.\tA\tC\t.\t.\t.\tGT:UET:UOPS\t0/1:-1:-1\t1|0:0:3"]


def test_crlf_and_no_format_pass_through():
    text = b"1\t10\t.\tA\tC\t.\t.\t.\r\n1\t11\t.\tA\tC\t.\t.\t.\tGT\t0/1\r\n"
    dec = vcfio.HostDecoder()
    dec.lines(np.frombuffer(text, dtype=np.uint8))
    out, bad = dec.rewrite(np.zeros(3, dtype=np.int64), np.zeros(0, dtype=L.VCF_EDIT_DTYPE), 1)
    assert out.tobytes() == b"1\t10\t.\tA\tC\t.\t.\t.\n1\t11\t.\tA\tC\t.\t.\t.\tGT:UOPS:UET\t0/1:-1:-1\n"


def test_line_status():
    _, bad = rewrite(["1\t10\t.\tA\tC\t.\t.\t.\tGT\t0/1\t0/1\t0/1"], 2)
    assert bad.tolist() == [L.VCFOUT_COLUMNS]
    _, bad = rewrite(["1\t10\t.\tA\tC\t.\t.\t.\tGT\t1\t0/1"], 2, {0: [(0, 1, 1, 0)]})
    assert bad.tolist() == [L.VCFOUT_HAPLOID]
    out, bad = rewrite(["1\t10\t.\tA\tC\t.\t.\t.\tGT\t1\t0/1"], 2, {0: [(0, 0, 1, 0)]})   # haploid, not phased
    assert not bad.any() and out[0].endswith("\t1:1:0\t0/1:-1:-1")
    _, bad = rewrite(["1\t10\t.\tA\tC\t.\t.\t.\tGT\t0/1:3\t0/1"], 2)
    assert bad.tolist() == [L.VCFOUT_FIELDS]


# ------------------------------------------------------------------------------------------------
# the driver: records -> edits, header, errors, containers
# ------------------------------------------------------------------------------------------------

def _record(chrom, start, end, kid="k", dad="d", mom="m", vartype="POINT", n_dad=0, n_mom=0):
    return {"region": {"chrom": chrom, "start": start, "end": end}, "kid": kid, "dad": dad, "mom": mom,
            "vartype": vartype, "evidence_type": "READBACKED", "dad_sites": ["s%d" % i for i in range(n_dad)],
            "mom_sites": ["t%d" % i for i in range(n_mom)], "dad_reads": ["r%d" % i for i in range(n_dad)],
            "mom_reads": ["q%d" % i for i in range(n_mom)], "cnv_dad_sites": [], "cnv_mom_sites": []}


def _write(tmp_path, text, name="in.vcf"):
    p = str(tmp_path / name)
    with (gzip.open(p, "wb") if name.endswith(".gz") else open(p, "wb")) as f:
        f.write(text.encode())
    return p


def _run(tmp_path, text, records, include_ambiguous=False, out="out.vcf", name="in.vcf"):
    p = _write(tmp_path, text, name)
    o = str(tmp_path / out)
    vcfio.write_phased_vcf(p, records, include_ambiguous, False, o, 10)
    return o


def test_duplicate_lines_svtype_and_ambiguous_records(tmp_path):
    body = ("1\t101\t.\tA\tC\t.\t.\t.\tGT\t0/1\t0/0\t0/0\n"
            "1\t101\t.\tA\tC\t.\t.\t.\tGT\t0/1\t0/0\t0/0\n"
            "1\t201\t.\tN\t<DEL>\t.\t.\tSVTYPE=DEL;END=500\tGT\t1/1\t0/0\t0/0\n"
            "1\t301\t.\tA\tC\t.\t.\t.\tGT\t0/1\t0/0\t0/0\n"
            "1\t401\t.\tA\tC\t.\t.\t.\tGT\t0/0\t0/0\t0/0\n")
    recs = {"1_100_101_k_POINT": _record("1", 100, 101, n_dad=3), "1_200_500_k_DEL": _record("1", 200, 500, "k",
            vartype="DEL", n_mom=4), "1_300_301_k_POINT": _record("1", 300, 301, n_dad=2, n_mom=2),
            "1_400_401_k_POINT": _record("1", 400, 401, n_dad=5)}
    text = HEAD + _cols("kdm") + body
    for amb in (False, True):
        lines = open(_run(tmp_path, text, copy.deepcopy(recs), amb)).read().split("\n")
        b = [l.split("\t", 9)[8:] for l in lines if l and not l.startswith("#")]
        assert b[0] == b[1] == ["GT:UOPS:UET", "1|0:3:0\t0/0:-1:-1\t0/0:-1:-1"]
        assert b[2] == ["GT:UOPS:UET", "0|1:4:0\t0/0:-1:-1\t0/0:-1:-1"]
        # dad and mom both with reads: ambiguous (dad|mom), written only with include_ambiguous, GT kept
        assert b[3] == ["GT:UOPS:UET", ("0/1:4:3" if amb else "0/1:-1:-1") + "\t0/0:-1:-1\t0/0:-1:-1"]
        assert b[4] == ["GT:UOPS:UET", "0/0:-1:-1\t0/0:-1:-1\t0/0:-1:-1"]      # a record, but no carrier


def test_header_rules(tmp_path):
    recs = {}
    body = "1\t101\t.\tA\tC\t.\t.\t.\tGT\t0/1\n"
    head = open(_run(tmp_path, HEAD + "##contig=<ID=1>\r\n" + _cols("k") + body, recs)).read().split("\n")
    assert head[:3] == ["##fileformat=VCFv4.2", vcfio.PASS_LINE, "##contig=<ID=1>"]
    has = HEAD + '##FILTER=<ID=PASS,Description="All filters passed">\n##FORMAT=<ID=UET,Number=1,Type=Float,' \
                 'Description="x">\n' + _cols("k")
    head = open(_run(tmp_path, has + body, recs)).read().split("\n")
    assert head.count(vcfio.PASS_LINE) == 1 and sum(h.startswith("##FORMAT=<ID=UET") for h in head) == 1
    assert head[3].startswith("##unfazed=") and head[4] == vcfio.UOPS_LINE and head[5].startswith("#CHROM")
    # a re-run: the unfazed line is added again, the FORMAT lines are not
    first = _run(tmp_path, HEAD + _cols("k") + body, {"1_100_101_k_POINT": _record("1", 100, 101, n_dad=1)},
                 out="first.vcf")
    again = str(tmp_path / "again.vcf")
    vcfio.write_phased_vcf(first, {"1_100_101_k_POINT": _record("1", 100, 101, n_mom=2)}, False, False, again, 10)
    lines = open(again).read().split("\n")
    assert sum(l.startswith("##unfazed=") for l in lines) == 2
    assert sum(l.startswith("##FORMAT=<ID=UOPS") for l in lines) == 1
    assert lines[-2].split("\t")[8:] == ["GT:UOPS:UET", "0|1:2:0"]


def test_errors_name_file_line_and_sample(tmp_path):
    recs = {"1_100_101_k_POINT": _record("1", 100, 101, n_dad=3)}
    text = HEAD + _cols(["x", "k"]) + "1\t50\t.\tA\tC\t.\t.\t.\tGT\t0\t0\n1\t101\t.\tA\tC\t.\t.\t.\tGT\t0\t1\n"
    with pytest.raises(ValueError, match=r"in\.vcf, line 4: the haploid GT '1' of sample k cannot be phased"):
        _run(tmp_path, text, copy.deepcopy(recs))
    text = HEAD + _cols("k") + "1\t101\t.\tA\tC\t.\t.\t.\tGT\t0/1\t0/0\n"
    with pytest.raises(ValueError, match=r"line 3: more sample columns than header samples"):
        _run(tmp_path, text, copy.deepcopy(recs))


def _phased_text(tmp_path):
    recs = {"1_100_101_k_POINT": _record("1", 100, 101, n_dad=3)}
    text = HEAD + _cols("kdm") + "1\t101\t.\tA\tC\t.\t.\t.\tGT\t0/1\t0/0\t0/0\n1\t201\t.\tA\tC\t.\t.\t.\tGT\t0/0\t0/1\t0/0\n"
    return text, recs


def test_containers(tmp_path, capsysbinary):
    text, recs = _phased_text(tmp_path)
    plain = _run(tmp_path, text, copy.deepcopy(recs), name="in.vcf.gz", out="out.vcf")
    want = open(plain, "rb").read()
    assert want.split(b"\n")[-3].endswith(b"\t1|0:3:0\t0/0:-1:-1\t0/0:-1:-1")
    gz = _run(tmp_path, text, copy.deepcopy(recs), name="in.vcf.gz", out="out.vcf.gz")
    assert open(gz, "rb").read().endswith(bamio.BGZF_EOF)
    r = bamio.BgzfReader(gz)
    raw, eof = r.stream_from(0, 1 << 30)
    assert eof and raw.tobytes() == want
    assert [d["kid"] for d in vcfio.read_dnms(gz)] == ["k", "d"]
    vcfio.write_phased_vcf(_write(tmp_path, text), copy.deepcopy(recs), False, False, "/dev/stdout", 10)
    assert capsysbinary.readouterr().out == want


def test_routing_without_cyvcf2(tmp_path):
    text, recs = _phased_text(tmp_path)
    src = _write(tmp_path, text, "dnms.vcf.gz")
    out = str(tmp_path / "o.vcf")
    with mock.patch.dict(sys.modules, {"cyvcf2": None}):
        unfazed.write_vcf_output(src, copy.deepcopy(recs), False, False, out, 10)
        assert "1|0:3:0" in open(out).read()
        with pytest.raises(ImportError):
            unfazed.write_vcf_output(src, copy.deepcopy(recs), False, False, str(tmp_path / "o.bcf"), 10)
        bcf = str(tmp_path / "dnms.bcf")
        open(bcf, "wb").close()
        with pytest.raises(ImportError):
            unfazed.write_vcf_output(bcf, copy.deepcopy(recs), False, False, out, 10)
    assert os.path.exists(out)
