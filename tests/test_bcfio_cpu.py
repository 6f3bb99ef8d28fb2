"""CPU: the native BCF reader (bcfio) and CSI indexes -- round trips against the packer and the text reader, a BCF
assembled byte by byte from the specification, CSI queries against a brute-force scan (also past 2^29 bp), CSI-indexed
.vcf.gz and .bam through the existing readers, malformed input, routing without cyvcf2 and pysam, the DNM reader and
the record size."""
import copy
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

from oracle import fakes
from tests.golden_util import CASES as GOLDEN_CASES, load_case
from tests.test_vcfio_cpu import assert_tables_equal, dnm_regions, no_decoders  # noqa: F401  (fixture)
from unfazed_b200 import _lib as L
from unfazed_b200 import bamio, bcfio, datasource, packers, vcfio
from unfazed_b200.synth import SynthConfig, make_dataset

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "unfazed_sm100.h")


@pytest.fixture(scope="module", autouse=True)
def native_lib():
    if not os.path.exists(L.LIB_PATH):
        import __graft_entry__ as g
        g.build()


def round_trip(sites, regions, tmp_path, **opts):
    """write_bcf -> bcfio.read_sites must equal pack_sites over the stand-ins and vcfio.read_sites of write_vcf."""
    bcf, vcf = str(tmp_path / "s.bcf"), str(tmp_path / "s.vcf.gz")
    bcfio.write_bcf(sites, bcf, **opts)
    vcfio.write_vcf(sites, vcf, **opts)
    fakes.register_vcf("mem://rt", sites)
    want = packers.pack_sites(fakes.VCF("mem://rt"), sites.trios, regions)
    got = bcfio.read_sites(bcf, sites.trios, regions)
    assert_tables_equal(want, got)
    assert_tables_equal(vcfio.read_sites(vcf, sites.trios, regions), got)
    assert np.array_equal(want.gq.view(np.uint32), got.gq.view(np.uint32))
    return bcf, want, got


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_round_trip_golden(tmp_path, name):
    ds, _ = load_case(name)
    prefix = "chr" if ds.sites.contigs[0].startswith("chr") else ""
    _, want, _ = round_trip(ds.sites, dnm_regions(ds.dnms, prefix), tmp_path)
    assert want.n_rows > 100


def test_round_trip_noisy_dataset_all_widths(tmp_path):
    ds = make_dataset(SynthConfig(dnms_per_trio=12, seed=41, n_trios=2, indel_frac=0.3, sv_frac=0.2, sv_max_len=30000))
    s = copy.deepcopy(ds.sites)
    rng = np.random.default_rng(5)
    s.gq[:, rng.random(s.n_rows) < 0.3] = rng.uniform(0, 99, size=(3, 1)).astype(np.float32)
    s.gq[0, ::7] = np.float32(1.0) / np.float32(3.0)
    s.gt[1, ::5] = 2
    s.rd[2, ::11] = -1
    s.ad[0, ::13] = -1
    s.rd[1, ::19] = 300                                 # int16 depths
    s.ad[2, ::23] = 70000                               # int32 depths
    for r in range(0, s.n_rows, 17):
        s.extras[r] = ("AC", ["A", "ACT"]) if r % 2 else ("G", ["*"])
        s.flag[r] = 0
    view, g_lo, _ = vcfio._records(s)
    n_rec = g_lo.shape[0] - 1
    orders = [("GT", "AD", "GQ"), ("GQ", "GT", "AD"), ("AD", "GQ", "GT")]
    fmt = [orders[g % 3] for g in range(n_rec)]
    path, want, _ = round_trip(s, dnm_regions(ds.dnms, ""), tmp_path, format_order=fmt)
    assert np.any(want.gq != np.round(want.gq)) and np.any(want.gt == 2) and len(want.extras) > 5
    bf = bcfio.BcfFile(path)
    buf, offs, _ = bf.fetch_union([(0, 0, 1 << 30)])
    recs = bcfio.HostDecoder().records(buf, offs, bf.keys, len(bf.samples))
    assert {1, 2, 3} <= set((recs["fmt_ct"][:, 2] & 15).tolist())       # AD as int8, int16 and int32


def test_round_trip_200_trio_cohort(tmp_path):
    ds = make_dataset(SynthConfig(n_trios=200, dnms_per_trio=1, seed=7, coverage=2.0, search_dist=2000))
    _, want, _ = round_trip(ds.sites, dnm_regions(ds.dnms, "", 2000), tmp_path)
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


# ---- a BCF assembled byte by byte from the specification (no code shared with write_bcf) ---------------------------

def bgzf(raw):
    """One BGZF block of raw (< 64 KiB): a gzip member with the BC extra subfield holding the block size - 1."""
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    cdata = co.compress(raw) + co.flush()
    return (b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", 25 + len(cdata))
            + cdata + struct.pack("<II", zlib.crc32(raw), len(raw)))


EOF_BLOCK = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
INT8, INT16, INT32, FLOAT, CHAR = 1, 2, 3, 5, 7
FMT = {INT8: "<b", INT16: "<h", INT32: "<i", FLOAT: "<f"}
M8, E8, M16, E16, M32, E32 = -128, -127, -32768, -32767, -2 ** 31, -2 ** 31 + 1
FMISS, FEOV = "fmiss", "feov"


def th(typ, n):
    """A type byte; a count of 15 or more follows as a typed int8 / int16."""
    if n < 15:
        return bytes([n << 4 | typ])
    return bytes([0xF0 | typ]) + (b"\x11" + struct.pack("<b", n) if n < 128 else b"\x12" + struct.pack("<h", n))


def vals(typ, xs):
    out = b""
    for x in xs:
        if x == FMISS:
            out += struct.pack("<I", 0x7F800001)
        elif x == FEOV:
            out += struct.pack("<I", 0x7F800002)
        else:
            out += struct.pack(FMT[typ], x)
    return out


def key(k):
    return b"\x11" + struct.pack("<b", k)


def text(s):
    return th(CHAR, len(s)) + s.encode()


def record(chrom, pos0, rlen, alleles, n_sample, info=(), fmt=(), n_sample_field=None):
    """info: [(key, typed bytes)]; fmt: [(key, type, count, [values of sample 0..n-1, count each])]."""
    shared = struct.pack("<iiiI", chrom, pos0, rlen, 0x7F800001)
    shared += struct.pack("<I", len(alleles) << 16 | len(info))
    shared += struct.pack("<I", len(fmt) << 24 | (n_sample if n_sample_field is None else n_sample_field))
    shared += text(".") + b"".join(text(a) for a in alleles) + th(INT8, 1) + b"\x00"
    shared += b"".join(key(k) + v for k, v in info)
    indiv = b""
    for k, typ, cnt, xs in fmt:
        flat = [x for sample in xs for x in sample]
        assert len(flat) == cnt * n_sample
        indiv += key(k) + th(typ, cnt) + vals(typ, flat)
    return struct.pack("<II", len(shared), len(indiv)) + shared + indiv


def assemble(path, header, recs, tids, csi=True, compress=True, magic=b"BCF\x02\x02"):
    """The file (header in one block, records in the next) and a CSI with one root-bin chunk per reference."""
    htext = header.encode() + b"\0"
    head = magic + struct.pack("<I", len(htext)) + htext
    body = b"".join(recs)
    if not compress:
        open(path, "wb").write(head + body)
        return
    b0 = bgzf(head)
    open(path, "wb").write(b0 + bgzf(body) + EOF_BLOCK)
    if not csi:
        return
    starts = np.cumsum([0] + [len(r) for r in recs])
    refs = b""
    n_ref = max(tids) + 1
    for t in range(n_ref):
        ix = [i for i, x in enumerate(tids) if x == t]
        if not ix:
            refs += struct.pack("<i", 0)
            continue
        vb, ve = (len(b0) << 16) | int(starts[ix[0]]), (len(b0) << 16) | int(starts[ix[-1] + 1])
        refs += struct.pack("<iIQi", 1, 0, vb, 1) + struct.pack("<QQ", vb, ve)
    idx = b"CSI\x01" + struct.pack("<iiii", 14, 5, 0, n_ref) + refs
    open(path + ".csi", "wb").write(bgzf(idx) + EOF_BLOCK)


SAMPLES = ["s0", "s1", "s2"]
LINE = "\t".join(["#CHROM", "POS", "ID", "REF", "ALT", "QUAL", "FILTER", "INFO", "FORMAT"] + SAMPLES) + "\n"
# header with IDX= (htslib's output) and header without (PASS at 0 implied, numbered by first appearance)
HEAD_IDX = ("##fileformat=VCFv4.2\n##FILTER=<ID=PASS,Description=\"All filters passed\",IDX=0>\n"
            "##INFO=<ID=DP,Number=1,Type=Integer,Description=\"depth, total\",IDX=7>\n"
            "##FORMAT=<ID=PL,Number=G,Type=Integer,Description=\"pl\",IDX=3>\n"
            "##FORMAT=<ID=GT,Number=1,Type=String,Description=\"g\",IDX=1>\n"
            "##FORMAT=<ID=GQ,Number=1,Type=Integer,Description=\"q\",IDX=5>\n"
            "##FORMAT=<ID=AD,Number=R,Type=Integer,Description=\"a\",IDX=2>\n"
            "##FORMAT=<ID=RO,Number=1,Type=Integer,Description=\"r\",IDX=8>\n"
            "##FORMAT=<ID=AO,Number=A,Type=Integer,Description=\"o\",IDX=9>\n"
            "##contig=<ID=1,length=1000000,IDX=1>\n##contig=<ID=2,length=1000000,IDX=0>\n" + LINE)
HEAD_PLAIN = ("##fileformat=VCFv4.2\n##INFO=<ID=DP,Number=1,Type=Integer,Description=\"d\">\n"
              "##FORMAT=<ID=GT,Number=1,Type=String,Description=\"g\">\n"
              "##FORMAT=<ID=GQ,Number=1,Type=Integer,Description=\"q\">\n"
              "##FORMAT=<ID=AD,Number=R,Type=Integer,Description=\"a\">\n"
              "##FORMAT=<ID=PL,Number=G,Type=Integer,Description=\"pl\">\n"
              "##FORMAT=<ID=RO,Number=1,Type=Integer,Description=\"r\">\n"
              "##FORMAT=<ID=AO,Number=A,Type=Integer,Description=\"o\">\n"
              "##contig=<ID=1>\n##contig=<ID=2>\n" + LINE)
KEYS = {"idx": dict(DP=7, PL=3, GT=1, GQ=5, AD=2, RO=8, AO=9, c1=1, c2=0),
        "plain": dict(DP=1, GT=2, GQ=3, AD=4, PL=5, RO=6, AO=7, c1=0, c2=1)}

# (pos0, alleles, expected [gt, gq, rd, ad] of s0, s1, s2); all records on contig "1" except the last
EXPECT = [
    (99, ["A", "C"], [(1, 30.0, 10, 300), (1, -1.0, -1, -1), (3, -1.0, 5, -1)]),
    (199, ["A", "C", "G"], [(1, 12.5, 1, 70002), (3, -1.0, 3, -1), (0, 7.0, -1, 9)]),
    (299, ["AT", "A"], [(2, -1.0, -1, -1)] * 3),
    (399, ["A", "C"], [(1, 99.0, 7, 7), (2, 100000.0, -1, -1), (3, -1.0, 2, 5)]),
    (49, ["G", "*"], [(2, -1.0, -1, -1), (1, -1.0, -1, -1), (0, -1.0, -1, -1)]),
]


def hand_records(k):
    pl = [[i * 17 + j for j in range(17)] for i in range(3)]          # 17 values per sample: a count overflow
    r1 = record(k["c1"], 99, 1, ["A", "C"], 3, info=[(k["DP"], th(INT8, 1) + b"\x09")], fmt=[
        (k["PL"], INT16, 17, pl),
        (k["GT"], INT8, 2, [[2, 4], [2, 5], [4, 4]]),                 # 0/1, 0|1, 1/1
        (k["GQ"], INT8, 1, [[30], [M8], [E8]]),
        (k["AD"], INT16, 2, [[10, 300], [M16, E16], [5, M16]])])
    r2 = record(k["c1"], 199, 1, ["A", "C", "G"], 3, fmt=[
        (k["GT"], INT8, 2, [[4, 6], [6, 6], [2, E8]]),                # 1/2, 2/2, haploid 0
        (k["GQ"], FLOAT, 1, [[12.5], [FMISS], [7.0]]),
        (k["AD"], INT32, 3, [[1, 2, 70000], [3, E32, E32], [M32, 4, 5]])])
    r3 = record(k["c1"], 299, 2, ["AT", "A"], 3)                       # n_fmt = 0
    r4 = record(k["c1"], 399, 1, ["A", "C"], 3, fmt=[
        (k["GT"], INT8, 3, [[2, 4, 4], [0, 0, E8], [4, E8, E8]]),       # triploid, ./., haploid 1
        (k["RO"], INT32, 1, [[7], [M32], [2]]),
        (k["AO"], INT16, 2, [[3, 4], [M16, E16], [5, E16]]),
        (k["GQ"], INT32, 1, [[99], [100000], [M32]])])
    r5 = record(k["c2"], 49, 1, ["G", "*"], 3, fmt=[
        (k["GT"], INT8, 2, [[0, 2], [0, 4], [3, 3]])])                # ./0, ./1, 0|0 (phase bit on the first)
    return [r1, r2, r3, r4], r5


def write_hand_bcf(path, variant="idx"):
    k = KEYS[variant]
    ones, r5 = hand_records(k)
    if k["c2"] < k["c1"]:
        assemble(path, HEAD_IDX, [r5] + ones, [0, 1, 1, 1, 1])
    else:
        assemble(path, HEAD_PLAIN, ones + [r5], [0, 0, 0, 0, 1])


@pytest.mark.parametrize("variant", ["idx", "plain"])
def test_hand_assembled_bcf(tmp_path, variant):
    path = str(tmp_path / "h.bcf")
    write_hand_bcf(path, variant)
    bf = bcfio.BcfFile(path)
    assert bf.samples == SAMPLES and bf.tids == {"1": KEYS[variant]["c1"], "2": KEYS[variant]["c2"]}
    got = bcfio.read_sites(path, [tuple(SAMPLES)], {"1": [(0, 1000)], "2": [(0, 1000)]})
    assert got.n_rows == 5 and got.pos.tolist() == [e[0] for e in EXPECT]
    assert got.flag.tolist() == [1, 0, 0, 1, 0]
    assert got.extras == {1: ("A", ["C", "G"]), 2: ("AT", ["A"]), 4: ("G", ["*"])}
    assert got.ref.tolist() == [ord(e[1][0][0]) for e in EXPECT] and got.alt.tolist() == [ord(e[1][1][0]) for e in EXPECT]
    for row, (_p, _al, cells) in enumerate(EXPECT):
        for m in range(3):
            have = (int(got.gt[m, row]), float(got.gq[m, row]), int(got.rd[m, row]), int(got.ad[m, row]))
            assert have == cells[m], (row, m, have, cells[m])
    # a query from the middle returns the overlapping records only
    assert bf.query("1", 200, 300)["pos0"].tolist() == [299]


# ---- CSI queries ------------------------------------------------------------------------------------------------

def _brute_force_queries(s, end, path, opener, rng, crossing=None):
    view, g_lo, g_contig = vcfio._records(s)
    f = opener(path)
    pos0 = np.array([int(s.pos[view[g_lo[g]]]) for g in range(g_lo.shape[0] - 1)])
    rend = np.array([end.get(g, p + len(s.ref_alts(int(view[g_lo[g]]))[0])) for g, p in enumerate(pos0)])
    hi = int(pos0.max()) + 10000
    for i in range(300):
        c = int(rng.integers(0, len(s.contigs)))
        a = int(rng.integers(-1000, hi)) if crossing is None or i % 2 else crossing - int(rng.integers(0, 200000))
        b = a + int(rng.integers(0, 400000 if crossing else 50000))
        a0, b0 = max(a, 0), max(b, a + 1, 1)
        want = np.flatnonzero((g_contig == c) & (pos0 < b0) & (rend > a0))
        got = f.query(s.contigs[c], a0, b0)
        assert got["pos0"].tolist() == pos0[want].tolist() and got["rend"].tolist() == rend[want].tolist()


def _with_ends(s, rng):
    view, g_lo, _ = vcfio._records(s)
    return {g: int(s.pos[view[g_lo[g]]]) + int(rng.integers(2, 300000)) for g in range(g_lo.shape[0] - 1)
            if rng.random() < 0.05}


def test_csi_queries_against_brute_force(tmp_path):
    ds, _ = load_case("sv_cnv")
    s = ds.sites
    rng = np.random.default_rng(9)
    end = _with_ends(s, rng)
    bcf, vcf = str(tmp_path / "q.bcf"), str(tmp_path / "q.vcf.gz")
    bcfio.write_bcf(s, bcf, end=end)
    vcfio.write_vcf(s, vcf, end=end, index="csi")
    assert bamio.CsiIndex(bcf + ".csi").depth == 5 and not os.path.exists(vcf + ".tbi")
    _brute_force_queries(s, end, bcf, bcfio.BcfFile, rng)
    _brute_force_queries(s, end, vcf, vcfio.VcfFile, rng)


def test_csi_queries_past_2_29_on_a_deeper_index(tmp_path):
    ds, _ = load_case("sv_cnv")
    s = copy.deepcopy(ds.sites)
    boundary = 1 << 29
    for b in range(s.n_blocks):
        lo, hi = int(s.blk_off[b]), int(s.blk_off[b + 1])
        if int(s.blk_contig[b]) == 0 and hi > lo:
            mid = int(s.pos[(lo + hi) // 2])
            s.pos[lo:hi] += np.int32(boundary - mid)          # records on both sides of 2^29
    rng = np.random.default_rng(4)
    end = _with_ends(s, rng)
    bcf, vcf = str(tmp_path / "d.bcf"), str(tmp_path / "d.vcf.gz")
    bcfio.write_bcf(s, bcf, end=end)
    vcfio.write_vcf(s, vcf, end=end, index="csi")
    assert bamio.CsiIndex(bcf + ".csi").depth == 6 and bamio.CsiIndex(vcf + ".csi").depth == 6
    _brute_force_queries(s, end, bcf, bcfio.BcfFile, rng, crossing=boundary)
    _brute_force_queries(s, end, vcf, vcfio.VcfFile, rng, crossing=boundary)


def test_csi_min_offset_follows_hts_itr_query(tmp_path):
    """The minimum offset is the loffset of the nearest existing bin at or left of beg's leaf bin towards the root;
    with it or without it (0) the records of a query are the same."""
    ds, _ = load_case("snv_noisy")
    path = str(tmp_path / "m.bcf")
    bcfio.write_bcf(ds.sites, path)
    bf = bcfio.BcfFile(path)
    idx = bf.csi
    c = ds.sites.contigs[0]
    tid = bf.tids[c]
    p = np.sort(bf.query(c, 0, 1 << 30)["pos0"])
    for beg in p[::7].tolist():
        leaf = bamio.bin_first(5) + (beg >> 14)
        b = leaf
        while b and b not in idx.loff[tid]:
            b = b - 1 if b > (((b - 1) >> 3) << 3) + 1 else (b - 1) >> 3
        assert idx.min_offset(tid, beg) == idx.loff[tid].get(b, 0)
        full = bf.query(c, beg, beg + 3000)
        saved = idx.min_offset
        idx.min_offset = lambda t, x: 0
        try:
            assert np.array_equal(bf.query(c, beg, beg + 3000), full)
        finally:
            idx.min_offset = saved


# ---- CSI through the existing readers ------------------------------------------------------------------------------

def test_vcf_gz_with_csi_equals_tbi(tmp_path):
    ds, _ = load_case("sexchrom_chr")
    reg = dnm_regions(ds.dnms, "chr")
    a, b = str(tmp_path / "t.vcf.gz"), str(tmp_path / "c.vcf.gz")
    vcfio.write_vcf(ds.sites, a)
    vcfio.write_vcf(ds.sites, b, index="csi")
    assert os.path.exists(b + ".csi") and not os.path.exists(b + ".tbi") and datasource.is_indexed_vcf(b)
    assert_tables_equal(vcfio.read_sites(a, ds.sites.trios, reg), vcfio.read_sites(b, ds.sites.trios, reg))


def test_bam_with_csi_equals_bai(tmp_path, no_decoders):
    from tests.test_bamio_cpu import CASES, _assert_tables_equal
    ds = make_dataset(CASES[1])
    tabs = []
    for index in ("bai", "csi"):
        d = tmp_path / index
        d.mkdir()
        dn = copy.deepcopy(ds.dnms)
        for kid in ds.reads.kids:
            bamio.write_bam(ds.reads, ds.reads.kids.index(kid), str(d / ("%s.bam" % kid)), index=index)
        for x in dn:
            x["bam"] = str(d / ("%s.bam" % x["kid"]))
        assert all(datasource.is_indexed_bam(x["bam"]) for x in dn)
        tabs.append(datasource.load_reads(dn, 5000, 151, 1000000))
    assert os.path.exists(str(tmp_path / "csi" / ("%s.bam.csi" % ds.reads.kids[0])))
    _assert_tables_equal(*tabs)
    # <stem>.csi is found too
    p = str(tmp_path / "csi" / ("%s.bam" % ds.reads.kids[0]))
    os.rename(p + ".csi", p[:-4] + ".csi")
    assert bamio.index_path(p) == p[:-4] + ".csi"


# ---- malformed input, routing ---------------------------------------------------------------------------------------

def _dnm_args():
    return [{"kid": "s0", "chrom": "1", "start": 100, "end": 101}], {"s0": {"dad": "s1", "mom": "s2"}}


def _malformed(path, kind):
    k = KEYS["plain"]
    ones, r5 = hand_records(k)
    recs, tids = ones + [r5], [0, 0, 0, 0, 1]
    if kind == "overrun":               # a GQ that claims 5 values per sample runs past l_indiv
        recs[0] = record(0, 99, 1, ["A", "C"], 3, fmt=[(k["GQ"], INT8, 1, [[1], [2], [3]])])
        recs[0] = recs[0][:-4] + th(INT8, 5) + recs[0][-3:]
    elif kind == "n_sample":
        recs[0] = record(0, 99, 1, ["A", "C"], 3, fmt=[(k["GT"], INT8, 2, [[2, 4]] * 3)], n_sample_field=4)
    elif kind == "type":
        recs[0] = record(0, 99, 1, ["A", "C"], 3, fmt=[(k["GQ"], INT8, 1, [[1], [2], [3]])])
        recs[0] = recs[0][:-4] + bytes([0x14]) + recs[0][-3:]
    elif kind == "reserved":
        recs[0] = record(0, 99, 1, ["A", "C"], 3, fmt=[(k["GQ"], INT8, 1, [[1], [-125], [3]])])
    elif kind == "overflow":
        recs[0] = record(0, 99, 1, ["A", "C"], 3, fmt=[(k["AD"], INT32, 3, [[1, 2 ** 31 - 1, 2 ** 31 - 1]] * 3)])
    assemble(path, HEAD_PLAIN, recs, tids, magic=b"XCF\x02\x02" if kind == "magic" else b"BCF\x02\x02")
    data = open(path, "rb").read()
    if kind == "crc":
        bs = struct.unpack_from("<H", data, 16)[0] + 1
        data = data[:bs - 8] + bytes([data[bs - 8] ^ 0xFF]) + data[bs - 7:]
    elif kind == "truncated":
        data = data[: len(data) // 2]
    elif kind == "no_eof":
        data = data[:-28]
    open(path, "wb").write(data)


@pytest.mark.parametrize("kind", ["overrun", "n_sample", "type", "reserved", "overflow", "magic", "crc", "truncated",
                                  "no_eof"])
def test_malformed_bcf_raises_through_load_sites(tmp_path, no_decoders, kind):
    path = str(tmp_path / ("%s.bcf" % kind))
    _malformed(path, kind)
    dnms, ped = _dnm_args()
    with pytest.raises(ValueError) as e:
        datasource.load_sites(path, dnms, ped, 5000)
    if kind in ("overrun", "n_sample", "type", "reserved", "overflow"):
        assert path in str(e.value) and "virtual offset" in str(e.value)


def test_load_sites_routes_bcf_without_cyvcf2(tmp_path, no_decoders):
    ds, _ = load_case("sexchrom_chr")
    bcf, vcf = str(tmp_path / "r.bcf"), str(tmp_path / "r.vcf.gz")
    bcfio.write_bcf(ds.sites, bcf)
    vcfio.write_vcf(ds.sites, vcf)
    assert datasource.is_indexed_bcf(bcf)
    assert_tables_equal(datasource.load_sites(vcf, ds.dnms, ds.pedigrees, 5000),
                        datasource.load_sites(bcf, ds.dnms, ds.pedigrees, 5000))
    # another BCF version, an uncompressed BCF and an unindexed BCF still go to cyvcf2 (unimportable here)
    other = str(tmp_path / "v21.bcf")
    assemble(other, HEAD_PLAIN, [hand_records(KEYS["plain"])[1]], [1], magic=b"BCF\x02\x01")
    plain = str(tmp_path / "plain.bcf")
    assemble(plain, HEAD_PLAIN, [hand_records(KEYS["plain"])[1]], [1], compress=False)
    open(plain + ".csi", "wb").write(open(other + ".csi", "rb").read())
    os.remove(bcf + ".csi")
    for p in (other, plain, bcf):
        assert not datasource.is_indexed_bcf(p)
        with pytest.raises(ImportError):
            datasource.load_sites(p, ds.dnms, ds.pedigrees, 5000)


# ---- DNM reader ----------------------------------------------------------------------------------------------------

DNM_TEXT = ["\t".join(["chr1", "1001", ".", "A", "G", ".", ".", ".", "GT", "0/1", "0/0", "./."]),
            "\t".join(["chr1", "5001", ".", "N", "<DEL>", ".", ".", "SVTYPE=DEL;END=9000", "GT", "0/0", "1/1", "0/1"]),
            "\t".join(["chr2", "301", ".", "C", "T", ".", ".", "SVLEN=4", "GT:GQ", "1|1:3", "0:1", "0|1:2"]),
            "\t".join(["chr2", "7001", ".", "N", "<DUP>", ".", ".", "END=7500;SVTYPE=DUP", "GT", "./1", "./0", "1"])]
DNM_HEAD = ("##fileformat=VCFv4.2\n##INFO=<ID=SVTYPE,Number=1,Type=String,Description=\"t\">\n"
            "##INFO=<ID=END,Number=1,Type=Integer,Description=\"e\">\n##INFO=<ID=SVLEN,Number=1,Type=Integer,Description=\"l\">\n"
            "##FORMAT=<ID=GT,Number=1,Type=String,Description=\"g\">\n##FORMAT=<ID=GQ,Number=1,Type=Integer,Description=\"q\">\n"
            "##contig=<ID=chr1>\n##contig=<ID=chr2>\n")


def dnm_bcf(path, samples, rows, contigs, compress=True):
    """A DNM BCF: rows of (contig index, pos0, end or None, ref, alt, svtype or None, GT codes per sample)."""
    head = ("##fileformat=VCFv4.2\n##INFO=<ID=SVTYPE,Number=1,Type=String,Description=\"t\">\n"
            "##INFO=<ID=END,Number=1,Type=Integer,Description=\"e\">\n"
            "##FORMAT=<ID=GT,Number=1,Type=String,Description=\"g\">\n" + "".join("##contig=<ID=%s>\n" % c
                                                                                for c in contigs)
            + "\t".join(["#CHROM", "POS", "ID", "REF", "ALT", "QUAL", "FILTER", "INFO", "FORMAT"] + samples) + "\n")
    recs = []
    for cid, p0, end, ref, alt, svt, gts in rows:
        info = []
        if svt is not None:
            info.append((1, text(svt)))
        if end is not None:
            info.append((2, b"\x13" + struct.pack("<i", end)))
        recs.append(record(cid, p0, (end - p0) if end is not None else len(ref), [ref, alt], len(samples), info=info,
                           fmt=[(3, INT8, 2, gts)]))
    assemble(path, head, recs, [r[0] for r in rows], csi=False, compress=compress)


def test_read_dnms_equals_text_reader(tmp_path, no_decoders):
    from unfazed_b200.unfazed import read_vars_vcf
    samples = ["k1", "k2", "k3"]
    txt = str(tmp_path / "d.vcf")
    with open(txt, "w") as f:
        f.write(DNM_HEAD + "\t".join(["#CHROM", "POS", "ID", "REF", "ALT", "QUAL", "FILTER", "INFO", "FORMAT"] + samples)
                + "\n" + "\n".join(DNM_TEXT) + "\n")
    want = list(vcfio.read_dnms(txt))
    assert len(want) == 7
    rows = [(0, 1000, None, "A", "G", None, [[2, 4], [2, 2], [0, 0]]),
            (0, 5000, 9000, "N", "<DEL>", "DEL", [[2, 2], [4, 4], [2, 4]]),
            (1, 300, None, "C", "T", None, [[4, 5], [2, -127], [2, 5]]),
            (1, 7000, 7500, "N", "<DUP>", "DUP", [[0, 4], [0, 2], [4, -127]])]
    for name, comp in (("d.bcf", True), ("u.bcf", False)):
        p = str(tmp_path / name)
        dnm_bcf(p, samples, rows, ["chr1", "chr2"], compress=comp)
        assert list(bcfio.read_dnms(p)) == want, name
        assert list(read_vars_vcf(p)) == want, name


def test_bcf_record_size_matches_header(tmp_path):
    prog = tmp_path / "bsize.c"
    prog.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){printf("%%zu %%zu %%zu\\n",'
                    'sizeof(UnfzBcfRec),offsetof(UnfzBcfRec,fmt_ct),offsetof(UnfzBcfRec,flags));return 0;}\n' % HEADER)
    exe = tmp_path / "bsize"
    subprocess.run(["gcc", str(prog), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got == [L.BCF_REC_DTYPE.itemsize, L.BCF_REC_DTYPE.fields["fmt_ct"][1], L.BCF_REC_DTYPE.fields["flags"][1]] \
        == [80, 56, 79]
