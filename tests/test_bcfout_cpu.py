"""CPU: the phased VCF writer of a BCF DNM list (bcfio.write_phased_vcf, csrc/bcfout.cu host entry points).
Hand-assembled records print the literal text of the formatting rules (DESIGN §5); random records written as BCF and as
VCF text (printed by a restatement of the rules kept here) give the same phased output through both writers; floats
equal Python's "%g"; malformed input raises; the header; the routing of unfazed.write_vcf_output without cyvcf2."""
import copy
import gzip
import re
import struct
import sys
from unittest import mock

import numpy as np
import pytest

from tests.test_bcfio_cpu import CHAR, E8, E16, E32, FLOAT, FMISS, FEOV, INT8, INT16, INT32, M8, M16, M32, assemble, \
    key, native_lib, text, th, vals  # noqa: F401  (fixture)
from tests.test_vcfout_cpu import _record
from unfazed_b200 import _lib as L
from unfazed_b200 import bamio, bcfio, unfazed, vcfio

COLS = ["#CHROM", "POS", "ID", "REF", "ALT", "QUAL", "FILTER", "INFO", "FORMAT"]
STRINGS = ["PASS", "q10", "LowQual", "DP", "AF", "DB", "STR", "SVTYPE", "GT", "GQ", "AD", "PL", "FT", "XF", "UOPS", "UET"]
ID = {k: i for i, k in enumerate(STRINGS)}
_KIND = {"DP": ("INFO", "Integer"), "AF": ("INFO", "Float"), "DB": ("INFO", "Flag"), "STR": ("INFO", "String"),
         "SVTYPE": ("INFO", "String"), "GT": ("FORMAT", "String"), "GQ": ("FORMAT", "Integer"),
         "AD": ("FORMAT", "Integer"), "PL": ("FORMAT", "Integer"), "FT": ("FORMAT", "String"),
         "XF": ("FORMAT", "Float"), "UOPS": ("FORMAT", "Float"), "UET": ("FORMAT", "Float")}


def header(samples, idx=True, uops=True):
    """A header declaring STRINGS in order (with IDX= as htslib writes BCF, or numbered by appearance) and chr1, chr2."""
    lines = ["##fileformat=VCFv4.2"]
    for i, k in enumerate(STRINGS):
        if not uops and k in ("UOPS", "UET"):
            continue
        x = ",IDX=%d" % i if idx else ""
        if k in ("PASS", "q10", "LowQual"):
            if k != "PASS" or idx:
                lines.append('##FILTER=<ID=%s,Description="f"%s>' % (k, x))
        else:
            kind, typ = _KIND[k]
            lines.append('##%s=<ID=%s,Number=.,Type=%s,Description="d, %s"%s>' % (kind, k, typ, k, x))
    lines += ["##contig=<ID=chr1,length=1000000%s>" % (",IDX=0" if idx else ""),
              "##contig=<ID=chr2%s>" % (",IDX=1" if idx else "")]
    return "\n".join(lines) + "\n" + "\t".join(COLS + list(samples)) + "\n"


def brec(chrom, pos0, alleles, n_sample, ident=".", qual=None, filters=(0,), info=(), fmt=(), rlen=None,
         n_sample_field=None):
    """One BCF record: ``qual`` a float or None (missing); ``filters`` dictionary ids; info [(key, typed bytes)];
    fmt [(key, type, count, [values of sample 0..n-1, count each; for strings one byte string of count bytes])]."""
    shared = struct.pack("<iii", chrom, pos0, len(alleles[0]) if rlen is None else rlen)
    shared += struct.pack("<I", 0x7F800001) if qual is None else struct.pack("<f", qual)
    shared += struct.pack("<I", len(alleles) << 16 | len(info))
    shared += struct.pack("<I", len(fmt) << 24 | (n_sample if n_sample_field is None else n_sample_field))
    shared += text(ident) + b"".join(text(a) for a in alleles)
    shared += th(INT8, len(filters)) + bytes(x & 0xFF for x in filters)
    shared += b"".join(key(k) + v for k, v in info)
    indiv = b""
    for k, typ, cnt, xs in fmt:
        flat = [x for sample in xs for x in sample]
        assert len(flat) == (1 if typ == CHAR else cnt) * n_sample
        indiv += key(k) + th(typ, cnt) + (b"".join(flat) if typ == CHAR else vals(typ, flat))
    return struct.pack("<II", len(shared), len(indiv)) + shared + indiv


def fmt_records(path, edits=None):
    """The records of an uncompressed BCF printed by the host entry points: (lines, record status)."""
    _text, samples, strs, contigs, buf, offs, where = bcfio._read_whole(path)
    dec = bcfio.HostDecoder()
    recs = bcfio._checked_records(dec, buf, offs, np.array([strs.get(k, -1) for k in bcfio.FORMAT_KEYS], np.int32),
                                  len(samples), where)
    rows = sorted((i, *e) for i, es in (edits or {}).items() for e in es)
    ed = np.zeros(len(rows), dtype=L.VCF_EDIT_DTYPE)
    for k, name in enumerate(("sample", "phase", "uops", "uet")):
        ed[name] = [r[k + 1] for r in rows]
    off = np.searchsorted(np.array([r[0] for r in rows], dtype=np.int64), np.arange(recs.shape[0] + 1)).astype(np.int64)
    fkeys = np.array([strs.get(k, -1) for k in ("GT", "UOPS", "UET")], dtype=np.int32)
    out, status = dec.format(off, ed, len(samples), bcfio.dictionaries(strs, contigs), fkeys)
    return out.tobytes().decode().split("\n")[:-1], status


def i8(*xs):
    return th(INT8, len(xs)) + vals(INT8, xs)


def hand_records():
    r1 = brec(0, 999, ["A", "C"], 3, ident="rs1", qual=50.0, filters=(1, 2), info=[
        (ID["DP"], th(INT16, 1) + vals(INT16, [300])), (ID["AF"], th(FLOAT, 2) + vals(FLOAT, [0.5, FMISS])),
        (ID["DB"], th(0, 0)), (ID["STR"], th(CHAR, 5) + b"abc\0\0")], fmt=[
        (ID["GT"], INT8, 2, [[2, 4], [2, 5], [4, 4]]),                       # 0/1, 0|1, 1/1
        (ID["GQ"], INT8, 1, [[30], [M8], [E8]]),                             # 30, missing, end of vector (empty)
        (ID["AD"], INT16, 2, [[10, 300], [M16, E16], [5, M16]]),
        (ID["PL"], INT32, 16, [list(range(16)), [M32] + [E32] * 15, [1, 2] + [E32] * 14]),   # a count of 16
        (ID["FT"], CHAR, 4, [[b"PASS"], [b"q\0\0\0"], [b"\0\0\0\0"]]),
        (ID["XF"], FLOAT, 1, [[1.5], [FMISS], [FEOV]])])
    r2 = brec(0, 1999, ["A", "C", "G"], 3, ident="", qual=0.1, filters=(), fmt=[
        (ID["UOPS"], INT8, 1, [[7], [M8], [1]]),
        (ID["GT"], INT8, 3, [[2, 4, 4], [0, 0, E8], [4, E8, E8]]),           # triploid, ./., haploid 1
        (ID["UET"], INT8, 1, [[0], [1], [2]])])
    r3 = brec(1, 49, ["G"], 3, info=[(ID["DP"], i8(3, M8, E8)), (ID["AF"], th(FLOAT, 1) + vals(FLOAT, [-2.25]))])
    r4 = brec(1, 99, ["AT", "A"], 3, qual=1e10, fmt=[
        (ID["GT"], INT16, 2, [[3, 5], [0, 2], [3, E16]]),                    # phase bit on the first, ./0, haploid 0
        (ID["XF"], FLOAT, 2, [[1e-7, 123456.5], [-0.0, 7.0], [FMISS, FEOV]])])
    return [r1, r2, r3, r4]


HAND_OUT = [
    "chr1\t1000\trs1\tA\tC\t50\tq10;LowQual\tDP=300;AF=0.5,.;DB;STR=abc\tGT:GQ:AD:PL:FT:XF:UOPS:UET"
    "\t1|0:30:10,300:0,1,2,3,4,5,6,7,8,9,10,11,12,13,14,15:PASS:1.5:4:0\t0|1:.:.:.:q:.:-1:-1\t1/1::5,.:1,2:::-1:-1",
    "chr1\t2000\t.\tA\tC,G\t0.1\t.\t.\tUOPS:GT:UET\t9:0|1|1:1\t-1:./.:-1\t-1:1:-1",
    "chr2\t50\t.\tG\t.\t.\tPASS\tDP=3,.;AF=-2.25\t.:UOPS:UET\t.:-1:-1\t.:-1:-1\t.:-1:-1",
    "chr2\t100\t.\tAT\tA\t1e+10\tPASS\t.\tGT:XF:UOPS:UET\t0|1:1e-07,123456:-1:-1\t./0:-0,7:-1:-1\t0:.:-1:-1",
]


def test_hand_records_print_the_rules(tmp_path):
    p = str(tmp_path / "h.bcf")
    assemble(p, header(["s0", "s1", "s2"]), hand_records(), [0, 0, 1, 1], compress=False)
    out, status = fmt_records(p, {0: [(0, 1, 4, 0)], 1: [(0, 2, 9, 1)]})
    assert out == HAND_OUT
    assert status.tolist() == [0, 0, 0, L.BCFOUT_FLOAT_HOST]       # 1e10 and 1e-07 are exponent style: the host's
    # without samples: no FORMAT column
    p0 = str(tmp_path / "n.bcf")
    assemble(p0, header([]), [brec(0, 5, ["A", "T"], 0)], [0], compress=False)
    assert fmt_records(p0)[0] == ["chr1\t6\t.\tA\tT\t.\tPASS\t."]


def test_line_status(tmp_path):
    p = str(tmp_path / "s.bcf")
    gt = [(ID["GT"], INT8, 2, [[4, E8], [2, 4]])]
    recs = [brec(0, 9, ["A", "C"], 2, fmt=gt), brec(0, 19, ["A", "C"], 2, info=[(40, i8(1))]),
            brec(5, 29, ["A", "C"], 2), brec(0, 39, ["A", "C"], 2, filters=(33,)),
            brec(0, 49, ["A", "C"], 2, fmt=[(ID["GT"], INT8, 1, [[-6], [2]])])]
    assemble(p, header(["a", "b"]), recs, [0, 0, 0, 0, 0], compress=False)
    out, status = fmt_records(p, {0: [(0, 1, 1, 0)]})
    assert status.tolist() == [L.BCFOUT_HAPLOID] + [L.BCFOUT_BAD] * 4 and out == []
    out, status = fmt_records(p, {0: [(0, 0, 1, 0)]})                    # haploid, not phased
    assert status[0] == 0


# ------------------------------------------------------------------------------------------------
# cross-path equality with the text writer
# ------------------------------------------------------------------------------------------------

def _g(x):
    return "%g" % float(np.float32(x))


def _vec_text(typ, xs):
    """A value vector as the rules print it (None missing, "E" end of vector; a str for strings)."""
    if typ == CHAR:
        return xs.split("\0")[0]
    out = []
    for x in xs:
        if x == "E":
            break
        out.append("." if x is None else (_g(x) if typ == FLOAT else str(x)))
    return ",".join(out)


def _gt_text(codes):
    out = ""
    for j, c in enumerate(codes):
        if c == "E":
            break
        if j:
            out += "/|"[c & 1]
        out += "." if c >> 1 == 0 else str((c >> 1) - 1)
    return out or "."


def _enc(typ, xs):
    if typ == CHAR:
        return xs.encode()
    m = {INT8: (M8, E8), INT16: (M16, E16), INT32: (M32, E32), FLOAT: (FMISS, FEOV)}[typ]
    return vals(typ, [m[0] if x is None else m[1] if x == "E" else x for x in xs])


FLOATS = [0.5, 12.25, 3.0, 99.5, 1e-3, 0.3333333, 123456.5, 2.5e7, 1e-6, -4.75]


def random_records(rng, samples, n_rec):
    """(BCF records, VCF text lines, phasing records): random ID / QUAL / FILTER / INFO, a random FORMAT layout with GT
    always present, missing values and ends of vector, ploidy 1-3, phased and missing alleles."""
    ns = len(samples)
    recs, lines, phasing = [], [], {}
    pos = 100
    for r in range(n_rec):
        pos += int(rng.integers(1, 50))
        chrom = int(rng.integers(0, 2))
        alleles = ["A", "C", "GT", "T"][: int(rng.integers(1, 5))]
        ident = ["", ".", "rs%d" % r][int(rng.integers(0, 3))]
        qual = None if rng.random() < 0.4 else float(np.float32(rng.choice(FLOATS)))
        filters = [[], [0], [1, 2], [2]][int(rng.integers(0, 4))]
        info_b, info_t = [], []
        sv = rng.random() < 0.2
        for k in rng.permutation(["DP", "AF", "DB", "STR"] + (["SVTYPE"] if sv else [])).tolist():
            if rng.random() < 0.5 and k != "SVTYPE":
                continue
            if k == "DP":
                xs = [int(x) for x in rng.integers(0, 40000, size=int(rng.integers(1, 4)))] + [None] * int(rng.integers(0, 2))
                info_b.append((ID[k], th(INT32, len(xs)) + _enc(INT32, xs)))
                info_t.append("DP=" + _vec_text(INT32, xs))
            elif k == "AF":
                xs = [float(np.float32(rng.choice(FLOATS))) for _ in range(int(rng.integers(1, 3)))]
                info_b.append((ID[k], th(FLOAT, len(xs)) + _enc(FLOAT, xs)))
                info_t.append("AF=" + _vec_text(FLOAT, xs))
            elif k == "DB":
                info_b.append((ID[k], th(0, 0)))
                info_t.append("DB")
            else:
                s = "DEL" if k == "SVTYPE" else "x%d" % r
                info_b.append((ID[k], text(s)))
                info_t.append("%s=%s" % (k, s))
        keys = ["GT"] + [k for k in ["GQ", "AD", "PL", "FT", "XF"] if rng.random() < 0.5]
        keys = [keys[i] for i in rng.permutation(len(keys))]
        fmt_b, cells = [], [[] for _ in range(ns)]
        gts = []
        for k in keys:
            if k == "GT":
                ploidy = int(rng.integers(1, 4))
                xs = []
                for s in range(ns):
                    n_al = ploidy if rng.random() < 0.8 else int(rng.integers(1, ploidy + 1))
                    codes = [int(rng.integers(0, len(alleles) + 1)) * 2 + int(rng.random() < 0.3) for _ in range(n_al)]
                    codes = [c if rng.random() < 0.9 else c & 1 for c in codes]
                    xs.append(codes + ["E"] * (ploidy - n_al))
                typ, cnt = INT8, ploidy
                gts = xs
            elif k == "FT":
                cnt, typ = 3, CHAR
                xs = [["PASS"[: int(rng.integers(0, 4))].ljust(3, "\0")] for _ in range(ns)]
            else:
                typ = {"GQ": [INT8, INT16][int(rng.integers(0, 2))], "AD": INT16, "PL": INT32, "XF": FLOAT}[k]
                cnt = {"GQ": 1, "AD": 2, "PL": int(rng.integers(1, 18)), "XF": 1}[k]
                lim = {INT8: 100, INT16: 30000, INT32: 1 << 30, FLOAT: 1}[typ]
                xs = []
                for s in range(ns):
                    v = [float(np.float32(rng.choice(FLOATS))) if typ == FLOAT else int(rng.integers(-lim // 2, lim))
                         for _ in range(cnt)]
                    v = [None if rng.random() < 0.1 else x for x in v]
                    cut = cnt if rng.random() < 0.7 else int(rng.integers(0, cnt + 1))
                    xs.append(v[:cut] + ["E"] * (cnt - cut))
            fmt_b.append((ID[k], typ, cnt, [_enc(typ, x[0] if typ == CHAR else x) for x in xs]))
            for s in range(ns):
                cells[s].append(_gt_text(xs[s]) if k == "GT" else _vec_text(typ, xs[s][0] if typ == CHAR else xs[s]))
        recs.append(_brec_raw(chrom, pos, alleles, ns, ident, qual, filters, info_b, fmt_b))
        names = ["chr1", "chr2"]
        lines.append("\t".join([names[chrom], str(pos + 1), ident or ".", alleles[0],
                                ",".join(alleles[1:]) or ".", "." if qual is None else _g(qual),
                                ";".join(STRINGS[f] for f in filters) or ".", ";".join(info_t) or ".", ":".join(keys)]
                               + [":".join(c) for c in cells]))
        for s in range(0, ns, 3):                                      # the kids
            codes = [c for c in gts[s] if c != "E"]
            al = [c >> 1 for c in codes]
            if len(codes) >= 2 and any(a >= 2 for a in al) and rng.random() < 0.8:
                o = int(rng.integers(0, 3))
                phasing["%s_%d_%d_%s_%s" % (names[chrom], pos, pos + 1, samples[s], "DEL" if sv else "POINT")] = \
                    _record(names[chrom], pos, pos + 1, samples[s], samples[s + 1], samples[s + 2],
                            "DEL" if sv else "POINT", n_dad=3 * (o != 1), n_mom=3 * (o != 0))
    return recs, lines, phasing


def _brec_raw(chrom, pos0, alleles, ns, ident, qual, filters, info, fmt):
    """brec with every sample's values of a FORMAT field given as one byte string."""
    r = brec(chrom, pos0, alleles, ns, ident=ident, qual=qual, filters=filters, info=info,
             fmt=[(k, INT8, 1, [[0]] * ns) for k, _t, _c, _x in fmt])
    l_shared = struct.unpack_from("<I", r)[0]
    indiv = b"".join(key(k) + th(t, c) + b"".join(xs) for k, t, c, xs in fmt)
    return struct.pack("<II", l_shared, len(indiv)) + r[8: 8 + l_shared] + indiv


def write_pair(tmp_path, rng, n_samples, n_rec, compress=True):
    samples = ["k%d" % (i // 3) if i % 3 == 0 else ("d%d" if i % 3 == 1 else "m%d") % (i // 3) for i in range(n_samples)]
    recs, lines, phasing = random_records(rng, samples, n_rec)
    order = sorted(range(n_rec), key=lambda i: (lines[i].split("\t")[0], i))
    recs, lines = [recs[i] for i in order], [lines[i] for i in order]
    bcf, vcf = str(tmp_path / "r.bcf"), str(tmp_path / "r.vcf")
    assemble(bcf, header(samples, idx=False, uops=False), recs, [int(l.startswith("chr2")) for l in lines], csi=False,
             compress=compress)
    with open(vcf, "w") as f:
        f.write(header(samples, idx=False, uops=False) + "\n".join(lines) + "\n")
    return bcf, vcf, phasing


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_bcf_writer_equals_text_writer(tmp_path, seed):
    rng = np.random.default_rng(seed)
    bcf, vcf, phasing = write_pair(tmp_path, rng, 12, 120, compress=bool(seed % 2))
    assert len(phasing) > 20
    for amb in (False, True):
        a, b = str(tmp_path / "t.vcf"), str(tmp_path / "b.vcf")
        vcfio.write_phased_vcf(vcf, copy.deepcopy(phasing), amb, False, a, 10)
        bcfio.write_phased_vcf(bcf, copy.deepcopy(phasing), amb, False, b, 10)
        got = open(b, "rb").read()
        assert got == open(a, "rb").read()
        assert got.count(b"1|0") and got.count(b"0|1")


# ------------------------------------------------------------------------------------------------
# floats
# ------------------------------------------------------------------------------------------------

def float_values(rng):
    xs = [np.float32(x) for x in (0.0, -0.0, 1.0, -3.0, 100000.0, 999999.0, 999999.5, 1e6, 1e-5, 1e-4, 123456.5, 123457.5,
                                  10000.25, 10000.75, 1000.125, 1000.375, 0.1, 2.5e-5, 16777216.0, 3.4e38)]
    for c in (1e-5, 1e-4, 1e6, 999999.5):
        f = np.float32(c)
        xs += [np.nextafter(f, np.float32(0)), np.nextafter(f, np.float32(np.inf))]
    xs += [np.float32(k) + np.float32(0.5) for k in rng.integers(100000, 999999, size=50)]     # 7th-digit ties
    xs += list(np.array([1, 2, 3, 77, 1 << 20, 1 << 12], dtype=np.uint32).view(np.float32))     # subnormals
    xs += list(rng.integers(-100000, 100000, size=50).astype(np.float32))                        # integers
    bits = rng.integers(0, 1 << 32, size=3000, dtype=np.uint64).astype(np.uint32)
    xs += [x for x in bits.view(np.float32) if np.isfinite(x)]
    xs += list((rng.standard_normal(500) * 10.0 ** rng.integers(-7, 8, size=500)).astype(np.float32))
    return [x for x in xs if (np.float32(x).view(np.uint32) & 0x7FFFFFFF) < 0x7F800000]


def test_floats_equal_python_g(tmp_path):
    xs = float_values(np.random.default_rng(3))
    fixed = ["e" not in "%g" % float(x) and (x == 0 or abs(x) >= np.finfo(np.float32).tiny) for x in xs]
    exact = [x for x, f in zip(xs, fixed) if f]
    host = [x for x, f in zip(xs, fixed) if not f]
    assert len(exact) > 500 and len(host) > 500
    p = str(tmp_path / "f.bcf")
    recs = [brec(0, 9 + i, ["A"], 0, info=[(ID["AF"], th(FLOAT, len(v)) + vals(FLOAT, [float(x) for x in v]))])
            for i, v in enumerate((exact, host))]
    assemble(p, header([]), recs, [0, 0], compress=False)
    out, status = fmt_records(p)
    for line, v in zip(out, (exact, host)):
        assert line.split("\t")[7] == "AF=" + ",".join("%g" % float(x) for x in v)
    # the exact integer path printed every value of the first record; the second needed the host's snprintf
    assert status.tolist() == [0, L.BCFOUT_FLOAT_HOST]


# ------------------------------------------------------------------------------------------------
# errors, header, containers, routing
# ------------------------------------------------------------------------------------------------

def _dnm_file(tmp_path, recs, name="d.bcf", samples=("k", "d", "m"), compress=True):
    p = str(tmp_path / name)
    assemble(p, header(list(samples)), recs, [0] * len(recs), csi=False, compress=compress)
    return p


GT3 = [(ID["GT"], INT8, 2, [[2, 4], [2, 2], [2, 2]])]
PHASING = {"chr1_100_101_k_POINT": _record("chr1", 100, 101, "k", "d", "m", n_dad=3)}


def test_errors_name_file_offset_and_sample(tmp_path):
    hap = [(ID["GT"], INT8, 2, [[4, E8], [2, 2], [2, 2]])]
    p = _dnm_file(tmp_path, [brec(0, 50, ["A", "C"], 3, fmt=GT3), brec(0, 100, ["A", "C"], 3, fmt=hap)])
    with pytest.raises(ValueError, match=r"d\.bcf, record at byte \d+: the haploid GT '1' of sample k cannot be phased"):
        bcfio.write_phased_vcf(p, copy.deepcopy(PHASING), False, False, str(tmp_path / "o.vcf"), 10)
    p = _dnm_file(tmp_path, [brec(0, 100, ["A", "C"], 3, fmt=GT3, info=[(60, i8(1))])], "bad.bcf")
    with pytest.raises(ValueError, match=r"bad\.bcf, record at byte \d+: malformed BCF record \(an id outside"):
        bcfio.write_phased_vcf(p, copy.deepcopy(PHASING), False, False, str(tmp_path / "o.vcf"), 10)
    p = _dnm_file(tmp_path, [brec(0, 100, ["A", "C"], 3, fmt=GT3, n_sample_field=4)], "ns.bcf")
    with pytest.raises(ValueError, match=r"ns\.bcf, record at byte \d+: malformed BCF record \(.*n_sample differs"):
        bcfio.write_phased_vcf(p, copy.deepcopy(PHASING), False, False, str(tmp_path / "o.vcf"), 10)


def test_header_drops_idx_and_adds_lines_once(tmp_path):
    p = _dnm_file(tmp_path, [brec(0, 100, ["A", "C"], 3, fmt=GT3)])
    o = str(tmp_path / "o.vcf")
    bcfio.write_phased_vcf(p, copy.deepcopy(PHASING), False, False, o, 10)
    lines = open(o).read().split("\n")
    head = [x for x in lines if x.startswith("#")]
    assert not any("IDX=" in x for x in head)
    assert head == vcfio.phased_header(re.sub(r",IDX=[0-9]+", "", header(["k", "d", "m"])).encode(),
                                       unfazed.__version__).decode().split("\n")[:-1]
    assert sum(x.startswith("##unfazed=") for x in head) == 1
    assert sum(x.startswith("##FORMAT=<ID=UOPS") for x in head) == 1 and sum(x.startswith("##FORMAT=<ID=UET")
                                                                          for x in head) == 1
    assert lines[-2] == "chr1\t101\t.\tA\tC\t.\tPASS\t.\tGT:UOPS:UET\t1|0:3:0\t0/0:-1:-1\t0/0:-1:-1"
    # without UOPS / UET in the header the two lines are added, before #CHROM
    p2 = str(tmp_path / "u.bcf")
    assemble(p2, header(["k", "d", "m"], uops=False), [brec(0, 100, ["A", "C"], 3, fmt=GT3)], [0], csi=False)
    bcfio.write_phased_vcf(p2, copy.deepcopy(PHASING), False, False, o, 10)
    head = [x for x in open(o).read().split("\n") if x.startswith("#")]
    assert head[-4].startswith("##unfazed=") and head[-3] == vcfio.UOPS_LINE and head[-2] == vcfio.UET_LINE


def test_routing_without_cyvcf2(tmp_path, capsysbinary):
    recs = [brec(0, 100, ["A", "C"], 3, fmt=GT3), brec(0, 200, ["A", "C"], 3, fmt=GT3)]
    srcs = [_dnm_file(tmp_path, recs, "dnms.bcf"), _dnm_file(tmp_path, recs, "plain.bcf", compress=False)]
    with mock.patch.dict(sys.modules, {"cyvcf2": None}):
        want = None
        for src in srcs:
            out = str(tmp_path / "o.vcf")
            unfazed.write_vcf_output(src, copy.deepcopy(PHASING), False, False, out, 10)
            got = open(out, "rb").read()
            assert want is None or got == want
            want = got
        assert want.split(b"\n")[-3].endswith(b"\t1|0:3:0\t0/0:-1:-1\t0/0:-1:-1")
        gz = str(tmp_path / "o.vcf.gz")
        unfazed.write_vcf_output(srcs[0], copy.deepcopy(PHASING), False, False, gz, 10)
        raw = open(gz, "rb").read()
        assert raw.endswith(bamio.BGZF_EOF) and gzip.decompress(raw) == want
        unfazed.write_vcf_output(srcs[0], copy.deepcopy(PHASING), False, False, "/dev/stdout", 10)
        assert capsysbinary.readouterr().out == want
        with pytest.raises(ImportError):                               # BCF output stays on cyvcf2
            unfazed.write_vcf_output(srcs[0], copy.deepcopy(PHASING), False, False, str(tmp_path / "o.bcf"), 10)
