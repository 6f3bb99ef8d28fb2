"""CPU: the native sites-VCF reader (vcfio) -- BGZF, TBI queries, the field decode of csrc/vcf.cu's host entry points,
and the SiteTable it builds, which must equal what packers.pack_sites builds from the cyvcf2 API (here the in-memory
fakes) over the same records, array for array."""
import copy
import gzip
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import fakes
from tests.golden_util import CASES as GOLDEN_CASES, load_case
from unfazed_b200 import _lib as L
from unfazed_b200 import datasource, packers, vcfio
from unfazed_b200.plan import strip_chr
from unfazed_b200.synth import SynthConfig, make_dataset

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "unfazed_sm100.h")
FIELDS = ("blk_trio", "blk_contig", "blk_off", "pos", "flag", "ref", "alt", "gt", "gq", "rd", "ad", "rec_id")


@pytest.fixture(scope="module", autouse=True)
def native_lib():
    if not os.path.exists(L.LIB_PATH):
        import __graft_entry__ as g
        g.build()


@pytest.fixture()
def no_decoders():
    """cyvcf2 and pysam unimportable; the registry empty."""
    saved = {m: sys.modules.get(m) for m in ("cyvcf2", "pysam")}
    datasource._registry.clear()
    sys.modules["cyvcf2"] = None
    sys.modules["pysam"] = None
    yield
    datasource._registry.clear()
    for m, v in saved.items():
        if v is None:
            sys.modules.pop(m, None)
        else:
            sys.modules[m] = v


def dnm_regions(dnms, prefix, search_dist=5000):
    """The regions datasource.load_sites asks for."""
    reg = {}
    for d in dnms:
        reg.setdefault(prefix + strip_chr(d["chrom"]), []).append((int(d["start"]) - search_dist - 2,
                                                                    int(d["end"]) + search_dist + 2))
    return reg


def assert_tables_equal(want, got):
    for f in FIELDS:
        a, b = getattr(want, f), getattr(got, f)
        assert a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a, b), f
    assert got.contigs == want.contigs and got.extras == want.extras and got.trios == want.trios


def round_trip(sites, regions, tmp_path, name="s.vcf.gz", **opts):
    path = str(tmp_path / name)
    vcfio.write_vcf(sites, path, **opts)
    fakes.register_vcf("mem://rt", sites)
    want = packers.pack_sites(fakes.VCF("mem://rt"), sites.trios, regions)
    got = vcfio.read_sites(path, sites.trios, regions)
    assert_tables_equal(want, got)
    return path, want, got


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_round_trip_golden(tmp_path, name):
    ds, _ = load_case(name)
    prefix = "chr" if ds.sites.contigs[0].startswith("chr") else ""
    _, want, _ = round_trip(ds.sites, dnm_regions(ds.dnms, prefix), tmp_path)
    assert want.n_rows > 100


def test_round_trip_noisy_dataset(tmp_path):
    ds = make_dataset(SynthConfig(dnms_per_trio=12, seed=41, n_trios=2, indel_frac=0.3, sv_frac=0.2, sv_max_len=30000))
    s = copy.deepcopy(ds.sites)
    rng = np.random.default_rng(5)
    # non-integral GQ (a Float GQ header), unknown GTs, missing depths, and non-simple records
    s.gq[:, rng.random(s.n_rows) < 0.3] = rng.uniform(0, 99, size=(3, 1)).astype(np.float32)
    s.gq[0, ::7] = np.float32(1.0) / np.float32(3.0)
    s.gt[1, ::5] = 2
    s.rd[2, ::11] = -1
    s.ad[0, ::13] = -1
    for r in range(0, s.n_rows, 17):
        s.extras[r] = ("AC", ["A", "ACT"]) if r % 2 else ("G", ["*"])
        s.flag[r] = 0
    path, want, got = round_trip(s, dnm_regions(ds.dnms, ""), tmp_path)
    assert vcfio.VcfFile(path).format_types["GQ"] == "Float"
    assert np.any(want.gq != np.round(want.gq)) and np.any(want.gt == 2) and len(want.extras) > 5


def test_round_trip_200_trio_cohort(tmp_path):
    ds = make_dataset(SynthConfig(n_trios=200, dnms_per_trio=1, seed=7, coverage=2.0, search_dist=2000))
    _, want, got = round_trip(ds.sites, dnm_regions(ds.dnms, "", 2000), tmp_path)
    assert len(set(want.blk_trio.tolist())) == 200


def test_round_trip_overlapping_abutting_negative_regions(tmp_path):
    ds, _ = load_case("snv_noisy")
    s = ds.sites
    c = s.contigs[0]
    p = s.pos[s.blk_off[0]: s.blk_off[1]].astype(int)
    a, b = int(p[3]), int(p[-5])
    regions = {c: [(a - 100, a + 500), (a + 200, a + 900), (a + 900, a + 1400), (b, b), (-50, 10), (b + 10, b + 11)]}
    for other in s.contigs[1:3]:
        regions[other] = [(-1000, 2000000000)]
    regions["nosuchcontig"] = [(0, 1000)]
    round_trip(s, regions, tmp_path)


# ---- hand-written text against a restatement of the decode contract -----------------------------------------------

def expect_sample(fmt, field, gq_type):
    """(gt_types, gt_quals, gt_ref_depths, gt_alt_depths) of one sample column, cyvcf2 0.31.0 defaults."""
    keys = fmt.split(":")
    vals = field.split(":")
    get = lambda k: vals[keys.index(k)] if k in keys and keys.index(k) < len(vals) else None
    gt = 2
    g = get("GT")
    if g is not None:
        al = g.replace("|", "/").split("/")
        a = None if al[0] == "." else int(al[0])
        if len(al) == 1:
            gt = 2 if a is None else {0: 0, 1: 3}.get(a, 2)
        else:
            b = None if al[1] == "." else int(al[1])
            if a is None and b is None:
                gt = 2
            elif a is None or b is None:
                gt = 2 if (a if a is not None else b) == 0 else 1
            else:
                gt = 1 if a != b else (0 if a == 0 else 3)
    q = get("GQ")
    gq = -1.0 if q in (None, ".") else float(np.float32(float(q)))
    num = lambda x: None if x == "." else int(x)
    if "AD" in keys:
        v = get("AD")
        parts = [] if v is None else [num(x) for x in v.split(",")]
        rd = -1 if not parts or parts[0] is None else parts[0]
        ad = -1 if len(parts) < 2 or any(x is None for x in parts[1:]) else sum(parts[1:])
    else:
        ro, ao = get("RO"), get("AO")
        rd = -1 if ro in (None, ".") else int(ro)
        aos = None if ao is None else [num(x) for x in ao.split(",")]
        ad = -1 if aos is None or any(x is None for x in aos) else sum(aos)
    return gt, gq, rd, ad


def write_text_vcf(tmp_path, samples, lines, gq_type="Integer", name="h.vcf.gz", contigs=("1",)):
    """A bgzipped VCF of these lines and its TBI (the index comes from the lines' CHROM / POS / REF / INFO END)."""
    head = "##fileformat=VCFv4.2\n" + "".join("##contig=<ID=%s>\n" % c for c in contigs)
    head += '##FORMAT=<ID=GQ,Number=1,Type=%s,Description="q">\n' % gq_type
    head += "\t".join(["#CHROM", "POS", "ID", "REF", "ALT", "QUAL", "FILTER", "INFO", "FORMAT"] + samples) + "\n"
    body = "".join(l + "\n" for l in lines).encode()
    path = str(tmp_path / name)
    from unfazed_b200.bamio import index_refs, write_bgzf
    import struct
    voff = write_bgzf(path, head.encode(), body)
    starts = np.cumsum([0] + [len(l) + 1 for l in lines]).astype(np.int64)
    tid, pos, end = [], [], []
    for l in lines:
        f = l.split("\t")
        tid.append(list(contigs).index(f[0]))
        p0 = int(f[1]) - 1 if f[1].isdigit() else 0
        e = p0 + len(f[3])
        for kv in (f[7].split(";") if len(f) > 7 else []):
            if kv.startswith("END=") and int(kv[4:]) > p0:
                e = int(kv[4:])
        pos.append(p0)
        end.append(e)
    names = b"".join(c.encode() + b"\0" for c in contigs)
    tbi = (b"TBI\x01" + struct.pack("<8i", len(contigs), 2, 1, 2, 0, ord("#"), 0, len(names)) + names
           + index_refs(len(contigs), np.array(tid), np.array(pos), np.array(end), voff(starts[:-1]), voff(starts[1:])))
    write_bgzf(path + ".tbi", tbi, b"")
    return path


HAND_FIELDS = [
    ("GT:AD:GQ", ["0/0:10,0:30", "0|1:5,6:12", "1/1:0,9:8", "1|0:.:.", "./.:.:.", "0:3,0:4", "1:0,4:5", "2:1,1:3",
                  "./1:2,.:7", "0/.:4,4:6", "./0:.,2:1", "1/2:1,2,3:50", "2/2:1,1,5:9", ".:3:2", "1/1", "0/1:8",
                  "0/1/1:3,4:5"]),
    ("GQ:GT:AD", ["30:0/0:10,0", ".:0/1:3,3", "12:1|1:.", "4", "5:./.", "7:0/1:.,.", "9:1/1:4"]),
    ("GT:GQ:RO:AO", ["0/1:20:5:6", "1/1:.:0:3,4", "0/0:15:.:.", "./.:1:2:.,1", "0/1:3:4"]),
    ("GT:RO:AD:AO:GQ", ["0/1:9:5,6:99:11", "0/0:9:.:99:12"]),
    ("AD:GQ", ["3,3:20", ".:."]),
]


@pytest.mark.parametrize("gq_type", ["Integer", "Float"])
def test_hand_written_fields(tmp_path, gq_type):
    vals = [f for _fmt, fs in HAND_FIELDS for f in fs]
    n = max(len(fs) for _fmt, fs in HAND_FIELDS)
    samples = ["s%d" % i for i in range(n)]
    lines = []
    for k, (fmt, fs) in enumerate(HAND_FIELDS):
        fs = list(fs)
        if gq_type == "Float":
            fs = [f.replace(":30", ":30.5").replace("20", "20.25").replace(":12", ":1.2e1") for f in fs]
        lines.append("\t".join(["1", str(100 + 10 * k), ".", "A", "C", ".", "PASS", ".", fmt] + fs))
    trios = [tuple(samples[i: i + 3]) for i in range(0, n - 2, 3)]
    path = write_text_vcf(tmp_path, samples, lines, gq_type)
    got = vcfio.read_sites(path, trios, {"1": [(0, 1000)]})
    assert got.n_rows == len(lines) * len(trios) and vals
    for row in range(got.n_rows):
        t = int(got.blk_trio[np.searchsorted(got.blk_off, row, side="right") - 1])
        k = int(got.rec_id[row])
        fmt = HAND_FIELDS[k][0]
        f = lines[k].split("\t")[9:]
        for m in range(3):
            s = samples.index(trios[t][m])
            field = f[s] if s < len(f) else None
            want = expect_sample(fmt, field, gq_type) if field is not None else (2, -1.0, -1, -1)
            have = (int(got.gt[m, row]), float(got.gq[m, row]), int(got.rd[m, row]), int(got.ad[m, row]))
            assert have == want, (fmt, field, have, want)


def test_hand_written_records(tmp_path):
    """REF / ALT classes, ALT '.' and '*', INFO END widening the overlap, a 3000-sample line, fewer sample columns."""
    samples = ["s%d" % i for i in range(3000)]
    big = ["0/1:%d,%d:%d" % (i % 50, i % 7, i % 99) for i in range(3000)]
    lines = [
        "\t".join(["1", "100", ".", "A", "G", ".", ".", "DP=3", "GT:AD:GQ"] + big),
        "\t".join(["1", "200", ".", "A", ".", ".", ".", ".", "GT"] + ["0/0"] * 3000),
        "\t".join(["1", "300", ".", "A", "*", ".", ".", ".", "GT"] + ["1/1"] * 3000),
        "\t".join(["1", "400", ".", "AT", "A", ".", ".", ".", "GT"] + ["0/1"] * 3000),
        "\t".join(["1", "500", ".", "N", "<DEL>", ".", ".", "SVTYPE=DEL;END=9000", "GT"] + ["0/1"] * 3000),
        "\t".join(["1", "600", ".", "C", "T,G", ".", ".", ".", "GT"] + ["1/2"] * 2),         # fewer columns
    ]
    path = write_text_vcf(tmp_path, samples, lines)
    trios = [("s0", "s1", "s2"), ("s2997", "s2998", "s2999")]
    # the SV's END reaches past 5000: a region there returns it; the SNV at 100 is not returned
    got = vcfio.read_sites(path, trios, {"1": [(5000, 5010)]})
    assert got.n_rows == 2 and set(got.pos.tolist()) == {499} and got.extras[0] == ("N", ["<DEL>"])
    got = vcfio.read_sites(path, trios, {"1": [(0, 10000)]})
    t1 = got.blk_off[1]
    assert got.pos[:t1].tolist() == [99, 199, 299, 399, 499, 599]
    assert got.flag[:t1].tolist() == [1, 0, 0, 0, 0, 0]
    assert got.extras[1] == ("A", []) and got.extras[2] == ("A", ["*"]) and got.extras[5] == ("C", ["T", "G"])
    assert got.ref[0] == ord("A") and got.alt[0] == ord("G") and got.alt[1] == 0
    assert got.gt[:, t1].tolist() == [1, 1, 1] and got.gq[:, t1].tolist() == [27.0, 28.0, 29.0]
    assert got.rd[:, t1].tolist() == [47, 48, 49] and got.ad[:, t1].tolist() == [1, 2, 3]
    # the line with two sample columns: the other samples are missing
    assert got.gt[:, 5].tolist() == [1, 1, 2] and got.gt[:, t1 + 5].tolist() == [2, 2, 2]


def test_malformed_lines_raise(tmp_path):
    good = "\t".join(["1", "100", ".", "A", "G", ".", ".", ".", "GT:GQ", "0/1:3", "0/1:3", "0/1:3"])
    bad = {"pos": good.replace("\t100\t", "\t1x0\t"), "columns": "1\t100\t.\tA\tG\t.\t.",
           "samples": good + "\t0/0:1", "overflow": good.replace("0/1:3\t0/1:3\t0/1:3", "0/1:3\t0/1:99999999999\t0/1:3")}
    for k, line in bad.items():
        path = write_text_vcf(tmp_path, ["a", "b", "c"], [line], name="%s.vcf.gz" % k)
        with pytest.raises(ValueError, match=r"%s.*virtual offset" % k):
            vcfio.read_sites(path, [("a", "b", "c")], {"1": [(0, 1000)]})


def test_float_gq_host_path_equals_fast_path(tmp_path):
    rng = np.random.default_rng(3)
    vals = ["%.*f" % (int(rng.integers(0, 6)), x) for x in rng.uniform(0, 100, 300)] + \
           ["1e-30", "3.4028235e38", "0.1234567890123456789", "1E2", "-0.0", "12345678901234567", "5e+1", "nan"]
    samples = ["s%d" % i for i in range(3)]
    lines = ["\t".join(["1", str(10 + i), ".", "A", "C", ".", ".", ".", "GQ"] + [v] * 3) for i, v in enumerate(vals)]
    path = write_text_vcf(tmp_path, samples, lines, "Float")
    fast = vcfio.read_sites(path, [tuple(samples)], {"1": [(0, 10000)]})
    slow = vcfio.read_sites(path, [tuple(samples)], {"1": [(0, 10000)]}, max_digits=0)
    want = np.array([np.float32(float(v)) for v in vals], dtype=np.float32)
    for t in (fast, slow):
        assert np.array_equal(t.gq[0], want, equal_nan=True)
        assert np.array_equal(t.gq.view(np.uint32), fast.gq.view(np.uint32))


# ---- queries, corruption, routing ------------------------------------------------------------------------------

def test_tbi_queries_against_brute_force(tmp_path):
    ds, _ = load_case("sv_cnv")
    s = ds.sites
    _view, g_lo, g_contig = vcfio._records(s)
    rng = np.random.default_rng(9)
    end = {g: int(s.pos[_view[g_lo[g]]]) + int(rng.integers(2, 300000)) for g in range(g_lo.shape[0] - 1)
           if rng.random() < 0.05}
    path = str(tmp_path / "q.vcf.gz")
    vcfio.write_vcf(s, path, end=end)
    vf = vcfio.VcfFile(path)
    pos0 = np.array([int(s.pos[_view[g_lo[g]]]) for g in range(g_lo.shape[0] - 1)])
    rend = np.array([end.get(g, p + len(s.ref_alts(int(_view[g_lo[g]]))[0])) for g, p in enumerate(pos0)])
    hi = int(pos0.max()) + 10000
    for _ in range(300):
        c = int(rng.integers(0, len(s.contigs)))
        a = int(rng.integers(-1000, hi))
        b = a + int(rng.integers(0, 50000))
        a0, b0 = max(a, 0), max(b, a + 1, 1)
        want = np.flatnonzero((g_contig == c) & (pos0 < b0) & (rend > a0))
        got = vf.query(s.contigs[c], a0, b0)
        assert got["pos0"].tolist() == pos0[want].tolist() and got["rend"].tolist() == rend[want].tolist()


def _corrupt_cases(path):
    data = open(path, "rb").read()
    crc = bytearray(data)
    bs = int.from_bytes(data[16:18], "little") + 1          # first block (the header)
    crc[bs - 8] ^= 0xFF
    return {"crc": bytes(crc), "truncated": data[: len(data) // 2], "no_eof": data[:-28]}


@pytest.mark.parametrize("kind", ["crc", "truncated", "no_eof"])
def test_corrupt_file_raises_through_load_sites(tmp_path, no_decoders, kind):
    ds, _ = load_case("snv_noisy")
    path = str(tmp_path / "c.vcf.gz")
    vcfio.write_vcf(ds.sites, path)
    data = _corrupt_cases(path)[kind]
    with open(path, "wb") as f:
        f.write(data)
    with pytest.raises(ValueError):
        datasource.load_sites(path, ds.dnms, ds.pedigrees, 5000)


def test_load_sites_routes_indexed_vcf_without_cyvcf2(tmp_path, no_decoders):
    ds, _ = load_case("sexchrom_chr")
    path = str(tmp_path / "r.vcf.gz")
    vcfio.write_vcf(ds.sites, path)
    got = datasource.load_sites(path, ds.dnms, ds.pedigrees, 5000)
    fakes.register_vcf("mem://r", ds.sites)
    trios = []
    for d in ds.dnms:
        t = (d["kid"], ds.pedigrees[d["kid"]]["dad"], ds.pedigrees[d["kid"]]["mom"])
        if t not in trios:
            trios.append(t)
    want = packers.pack_sites(fakes.VCF("mem://r"), trios, dnm_regions(ds.dnms, "chr"))
    assert_tables_equal(want, got)
    # an unindexed file still goes to cyvcf2 (unimportable here)
    os.remove(path + ".tbi")
    with pytest.raises(ImportError):
        datasource.load_sites(path, ds.dnms, ds.pedigrees, 5000)


def test_read_dnms_equals_bed_reader(tmp_path, no_decoders):
    from unfazed_b200.unfazed import read_vars_bed, read_vars_vcf
    samples = ["k1", "k2", "k3"]
    lines = ["\t".join(["chr1", "1001", ".", "A", "G", ".", ".", ".", "GT", "0/1", "0/0", "./."]),
             "\t".join(["chr1", "5001", ".", "N", "<DEL>", ".", ".", "SVTYPE=DEL;END=9000", "GT", "0/0", "1/1", "0/1"]),
             "\t".join(["chr2", "301", ".", "C", "T", ".", ".", "SVLEN=4", "GT:GQ", "1|1:3", "0:1", "0|1:2"]),
             "\t".join(["chr2", "7001", ".", "N", "<DUP>", ".", ".", "END=7500;SVTYPE=DUP", "GT", "./1", "./0", "1"])]
    text = "##fileformat=VCFv4.2\n" + "\t".join(["#CHROM", "POS", "ID", "REF", "ALT", "QUAL", "FILTER", "INFO",
                                                 "FORMAT"] + samples) + "\n" + "\n".join(lines) + "\n"
    bed_rows = [("chr1", 1000, 1001, "k1", "POINT"), ("chr1", 5000, 9000, "k2", "DEL"), ("chr1", 5000, 9000, "k3", "DEL"),
                ("chr2", 300, 301, "k1", "POINT"), ("chr2", 300, 301, "k3", "POINT"),
                ("chr2", 7000, 7500, "k1", "DUP"), ("chr2", 7000, 7500, "k3", "DUP")]
    bed = tmp_path / "d.bed"
    bed.write_text("".join("%s\t%d\t%d\t%s\t%s\n" % r for r in bed_rows))
    want = list(read_vars_bed(str(bed)))
    for name, opener in (("d.vcf", open), ("d.vcf.gz", gzip.open)):
        with opener(str(tmp_path / name), "wt") as f:
            f.write(text)
        assert list(read_vars_vcf(str(tmp_path / name))) == want, name
    plain = str(tmp_path / "b.vcf.gz")
    from unfazed_b200.bamio import write_bgzf
    write_bgzf(plain, text.encode(), b"")
    assert list(vcfio.read_dnms(plain)) == want


def test_native_prefix(tmp_path):
    for contig, want in (("chr7", "chr"), ("7", ""), ("CHR7", "CHR"), ("Chrom7", "Chr"), ("X", "")):
        path = write_text_vcf(tmp_path, ["a"], ["\t".join([contig, "5", ".", "A", "C", ".", ".", ".", "GT", "0/1"])],
                              name="p%s.vcf.gz" % contig, contigs=(contig,))
        assert vcfio.VcfFile(path).prefix == want
        fakes.register_vcf("mem://p", vcfio.read_sites(path, [], {contig: [(0, 10)]}))


def test_vcf_record_size_matches_header(tmp_path):
    prog = tmp_path / "vsize.c"
    prog.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){printf("%%zu %%zu %%zu\\n",'
                    'sizeof(UnfzVcfRec),offsetof(UnfzVcfRec,slot),offsetof(UnfzVcfRec,flags));return 0;}\n' % HEADER)
    exe = tmp_path / "vsize"
    subprocess.run(["gcc", str(prog), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got == [L.VCF_REC_DTYPE.itemsize, L.VCF_REC_DTYPE.fields["slot"][1], L.VCF_REC_DTYPE.fields["flags"][1]] \
        == [64, 56, 62]
