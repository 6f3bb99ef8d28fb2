"""CPU: the native CRAM 3.0 reader (cramio) -- the same reads written as CRAM and as BAM give the same records and the
same ReadTable; rANS 4x8, CRAI queries, malformed files and routing."""
import copy
import gzip
import os
import struct
import subprocess
import sys
import zlib

import numpy as np
import pytest

from oracle import fakes
from tests.test_bamio_cpu import _assert_tables_equal, modified
from unfazed_b200 import _lib as L
from unfazed_b200 import bamio, cramio, datasource
from unfazed_b200.schema import AUX_HAS_SA, QUAL_ESCAPE
from unfazed_b200.synth import SynthConfig, make_dataset

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "unfazed_sm100.h")

SMALL = [SynthConfig(dnms_per_trio=3, seed=401, coverage=10.0),
         SynthConfig(dnms_per_trio=3, seed=402, coverage=10.0, sv_frac=0.4, sv_max_len=20000, indel_frac=0.3),
         SynthConfig(dnms_per_trio=3, seed=403, coverage=10.0, chr_prefix="chr", sex_chrom_frac=0.3, male_frac=1.0)]


@pytest.fixture(scope="module", autouse=True)
def native_lib():
    if not os.path.exists(L.LIB_PATH):
        import __graft_entry__ as g
        g.build()


@pytest.fixture()
def clean_modules():
    datasource._registry.clear()
    yield
    datasource._registry.clear()
    for m in ("cyvcf2", "pysam"):
        if m in sys.modules and (sys.modules[m] is None or getattr(sys.modules[m], "__fake__", False)):
            del sys.modules[m]


def write_fasta(path, names, lens, seqs=None, seed=0, width=60):
    """A FASTA (and no .fai) with random ACGT sequences unless ``seqs`` gives them."""
    rng = np.random.default_rng(seed)
    with open(path, "w") as f:
        for i, (n, ln) in enumerate(zip(names, lens)):
            s = seqs[i] if seqs else np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, ln)].tobytes().decode()
            f.write(">%s some description\n" % n + "\n".join(s[k:k + width] for k in range(0, len(s), width)) + "\n")


def consensus_fasta(path, reads, kid, bam_path):
    """A reference whose bases are the first aligned read base at each position (random elsewhere): most read bases
    become matches."""
    f = bamio.BamFile(bam_path)
    rng = np.random.default_rng(1)
    seqs = []
    for tid, (name, ln) in enumerate(zip(f.refs, f.ref_lens)):
        s = rng.choice(np.frombuffer(b"ACGT", np.uint8), ln)
        buf, offs, rec = f.query(name, 0, ln)
        for o, r in zip(offs.tolist(), rec):
            if r["flag"] & 4:
                continue
            fx = cramio._bam_fields(buf, o)
            rp, gp = 0, fx["pos"]
            for w in fx["cigar"]:
                op, n = w & 15, w >> 4
                if op == 0:
                    seg = np.frombuffer(fx["seq"][rp:rp + n], np.uint8)
                    ok = np.isin(seg, np.frombuffer(b"ACGT", np.uint8))
                    s[gp:gp + n][ok] = seg[ok]
                if op in (0, 1, 4):
                    rp += n
                if op in (0, 2, 3):
                    gp += n
        seqs.append(s.tobytes().decode())
    write_fasta(path, f.refs, f.ref_lens, seqs)


def _all_records(cf):
    sl = sorted(set(zip(cf.crai[:, 3].tolist(), cf.crai[:, 4].tolist())))
    return cf.decode(sl)


def _write_pair(reads, k, tmp_path, ref=None, cram_opts=None, bam_opts=None, tag=""):
    bp = str(tmp_path / ("k%d%s.bam" % (k, tag)))
    bamio.write_bam(reads, k, bp, **(bam_opts or {}))
    if ref is None:
        f = bamio.BamFile(bp)
        ref = str(tmp_path / ("ref%d%s.fa" % (k, tag)))
        write_fasta(ref, f.refs, f.ref_lens, seed=k)
    cp = str(tmp_path / ("k%d%s.cram" % (k, tag)))
    cramio.write_cram(reads, k, cp, ref, **(cram_opts or {}), **(bam_opts or {}))
    return bp, cp, ref


def _regions(ds, reads, margin=6000):
    reg = {}
    for d in ds.dnms:
        for p in {int(d["start"]), int(d["end"])}:
            reg.setdefault(d["kid"], {}).setdefault(d["chrom"], []).append((p - margin, p + margin))
    return reg


def _kid_opts(reads, k, opts):
    if "extra_tags" not in opts:
        return opts
    rows = set(np.concatenate([np.arange(reads.blk_off[b], reads.blk_off[b + 1]) for b in range(reads.n_blocks)
                               if reads.blk_kid[b] == k] or [np.zeros(0, np.int64)]).tolist())
    o = dict(opts)
    o["extra_tags"] = {r: v for r, v in opts["extra_tags"].items() if r in rows}
    return o


def round_trip(ds, reads, tmp_path, cram_opts=None, bam_opts=None, consensus=False, tag=""):
    """read_regions over the CRAMs equals read_regions over the BAMs of the same reads, and every CRAM decodes to the
    BAM's record bytes."""
    bam_paths, crams = {}, {}
    for k, kid in enumerate(reads.kids):
        bo = _kid_opts(reads, k, bam_opts or {})
        ref = None
        if consensus:
            bp = str(tmp_path / ("c%d%s.bam" % (k, tag)))
            bamio.write_bam(reads, k, bp, **bo)
            ref = str(tmp_path / ("cons%d%s.fa" % (k, tag)))
            consensus_fasta(ref, reads, k, bp)
        bp, cp, ref = _write_pair(reads, k, tmp_path, ref, cram_opts, bo, tag)
        bam_paths[kid] = bp
        crams[kid] = cramio.CramFile(cp, ref)
        f = bamio.BamFile(bp)
        bbuf, _ = f.bgzf.stream_from(f.first_voff, 1 << 40)
        cbuf, coffs = _all_records(crams[kid])
        assert cbuf.tobytes() == bbuf.tobytes()
        assert np.array_equal(coffs, bamio.record_offsets(bbuf)[0])
    reg = _regions(ds, reads)
    want = bamio.read_regions(bam_paths, reg, head_reads=500)
    got = bamio.read_regions(crams, reg, head_reads=500)
    assert want.n_reads > 0
    _assert_tables_equal(want, got)
    return got


@pytest.mark.parametrize("cfg", SMALL, ids=[str(c.seed) for c in SMALL])
def test_round_trip_equals_bam(tmp_path, cfg):
    ds = make_dataset(cfg)
    round_trip(ds, ds.reads, tmp_path)


def noisy(ds, seed=12):
    """``modified`` plus unmapped reads placed at their mate (no CIGAR, MAPQ 0), secondary and supplementary flags,
    H / N / P operations, and an RG tag last (the RG data series)."""
    reads, opts = modified(ds, seed)
    t = reads
    rng = np.random.default_rng(seed)
    h = t.hdr
    paired = np.flatnonzero((h["mate"] >= 0) & (h["n_cigar"] == 1))
    um = paired[rng.random(paired.shape[0]) < 0.03]
    h["flag"][um] |= 0x4
    h["mapq"][um] = 0
    h["n_cigar"][um] = 0
    sec = np.flatnonzero(rng.random(t.n_reads) < 0.02)
    h["flag"][sec] |= np.where(rng.random(sec.shape[0]) < 0.5, 0x100, 0x800).astype(np.uint16)
    # a few single-M CIGARs gain hard clips, a reference skip or padding around an insertion
    cig = t.cigar.copy()
    one = np.flatnonzero((h["n_cigar"] == 1) & ((h["flag"] & 4) == 0))[:40]
    words, offs = [], []
    new = []
    for r in range(t.n_reads):
        o, n = int(h["cigar_off"][r]), int(h["n_cigar"][r])
        w = list(cig[o:o + n])
        if r in set(one.tolist()):
            ln = int(w[0] >> 4)
            kind = r % 3
            if kind == 0:
                w = [(5 << 4) | 5, w[0], (3 << 4) | 5]
            elif kind == 1:
                w = [((ln - 20) << 4) | 0, (100 << 4) | 3, (20 << 4) | 0]
            else:
                w = [((ln - 20) << 4) | 0, (2 << 4) | 6, (1 << 4) | 1, (2 << 4) | 6, (19 << 4) | 0]
        offs.append(len(words))
        words += w
        new.append(len(w))
    t.cigar = np.array(words, dtype=np.uint32)
    h["cigar_off"] = offs
    h["n_cigar"] = new
    object.__setattr__(t, "_ref_ends", None)
    opts["common_tags"] = bamio.encode_tag("RG", "Z", "grp1")
    return t, opts


def test_round_trip_noisy_every_method_and_encoding(tmp_path):
    ds = make_dataset(SMALL[0])
    reads, opts = noisy(ds)
    variants = [dict(), dict(method="raw", encoding="core"), dict(method="bzip2", records_per_slice=300, slices_per_container=4),
                dict(method="lzma", multi_ref=True, records_per_slice=2000), dict(method="rans0", embed_ref=True),
                dict(method="rans1", rr=False, encoding="core"),
                dict(method={"*": "gzip", "QS": "rans1", "BA": "rans0", "RN": "bzip2"}, records_per_slice=700)]
    for i, v in enumerate(variants):
        got = round_trip(ds, reads, tmp_path, cram_opts=v, bam_opts=opts, tag="v%d" % i)
    assert np.any(got.hdr["aux"] & AUX_HAS_SA) and np.any(got.qual & QUAL_ESCAPE)
    assert np.any(got.hdr["flag"] & 0x4) and np.any(got.hdr["flag"] & 0x900)


def test_round_trip_consensus_reference_and_encodings(tmp_path):
    ds = make_dataset(SMALL[1])
    reads, opts = noisy(ds, 5)
    for i, v in enumerate([dict(encoding="core"), dict(encoding="external")]):
        round_trip(ds, reads, tmp_path, cram_opts=v, bam_opts=opts, consensus=True, tag="c%d" % i)


def test_encodings_decode_what_the_writer_meant(tmp_path):
    """Each bit-stream encoding forced on the series it can hold."""
    ds = make_dataset(SMALL[0])
    reads = ds.reads
    E = cramio
    forced = [{"FP": (E.E_GAMMA, 1), "DL": (E.E_SUBEXP, 0, 1), "RL": (E.E_BETA, 0, 16), "MQ": (E.E_BETA, 0, 8)},
              {"FN": (E.E_SUBEXP, 0, 0), "FP": (E.E_SUBEXP, 0, 3), "RG": (E.E_GAMMA, 2),
               "RN": (E.E_BYTE_ARRAY_LEN, (E.E_HUFFMAN, list(range(1, 64)), [6] * 63), (E.E_EXTERNAL, 30))}]
    for i, f in enumerate(forced):
        round_trip(ds, reads, tmp_path, cram_opts=dict(encoding=f), tag="e%d" % i)


def test_huffman_canonical_codes():
    assert cramio.canonical_codes([65, 66, 67, 68], [1, 2, 3, 3]) == [(0, 1, 65), (2, 2, 66), (6, 3, 67), (7, 3, 68)]
    assert cramio.canonical_codes([5], [0]) == [(0, 0, 5)]


@pytest.mark.parametrize("order", [0, 1])
def test_rans4x8_round_trips(order):
    rng = np.random.default_rng(order)
    big = bytes(rng.choice(np.frombuffer(b"ACGTN", np.uint8), 1_100_000, p=[0.3, 0.2, 0.2, 0.29, 0.01]))
    for data in (b"", b"x", b"q" * 1000, bytes(range(256)) * 5 + b"tail", rng.bytes(4099), big):
        assert cramio.rans_decode(cramio.rans_encode(data, order)) == data
    enc = bytearray(cramio.rans_encode(big, order))
    with pytest.raises(ValueError):
        cramio.rans_decode(bytes(enc[: len(enc) // 2]))


def test_crai_queries_equal_brute_force_scan(tmp_path):
    ds = make_dataset(SMALL[1])
    _, cp, ref = _write_pair(ds.reads, 0, tmp_path, cram_opts=dict(records_per_slice=150, slices_per_container=3))
    cf = cramio.CramFile(cp, ref)
    buf, offs = _all_records(cf)
    rec = bamio.parse_records(buf, offs)
    keys = [buf[o:o + 4 + int(buf[o:o + 4].view("<i4")[0])].tobytes() for o in offs.tolist()]
    rng = np.random.default_rng(5)
    n_checked = 0
    for it in range(300):
        tid = int(rng.integers(0, len(cf.refs)))
        ln = cf.ref_lens[tid]
        kind = it % 4
        if kind == 0:
            beg = end = int(rng.integers(0, ln))
        elif kind == 1:
            beg, end = max(0, ln - int(rng.integers(1, 3000))), ln
        else:
            beg = int(rng.integers(0, ln))
            end = beg + int(rng.integers(1, 40000))
        qb, qo = cf.fetch_union([(tid, beg, end)])
        qr = bamio.parse_records(qb, qo)
        keep = (qr["ref_id"] == tid) & (qr["pos"] < end) & (qr["end"] > beg)
        got = [qb[o:o + 4 + int(qb[o:o + 4].view("<i4")[0])].tobytes() for o in qo[keep].tolist()]
        want = np.flatnonzero((rec["ref_id"] == tid) & (rec["pos"] < end) & (rec["end"] > max(beg, 0)))
        assert got == [keys[i] for i in want.tolist()], (tid, beg, end)
        n_checked += want.shape[0]
    assert n_checked > 0


def _patch_block(path, out, find, edit):
    """A copy of the CRAM with one block's data edited (``edit(data) -> data`` of the first block whose raw data contain
    ``find``) and its CRC32 recomputed."""
    raw = bytearray(open(path, "rb").read())
    p = raw.index(find)
    # walk back to the block start: blocks here are raw, so the data start right after the ITF8 header fields
    for s in range(p - 1, max(p - 64, 0), -1):
        try:
            r = cramio._Reader(raw, s)
            method, ctype, cid, size, rsize = r.byte(), r.byte(), r.itf8(), r.itf8(), r.itf8()
        except cramio._Short:
            continue
        if method == 0 and ctype in (1, 2) and size == rsize and r.p <= p < r.p + size:
            crc = struct.unpack_from("<I", raw, r.p + size)[0]
            if zlib.crc32(bytes(raw[s:r.p + size])) == crc:
                data = edit(bytes(raw[r.p:r.p + size]))
                assert len(data) == size
                raw[r.p:r.p + size] = data
                raw[r.p + size:r.p + size + 4] = struct.pack("<I", zlib.crc32(bytes(raw[s:r.p + size])))
                open(out, "wb").write(bytes(raw))
                return
    raise AssertionError("block not found")


def test_malformed_files_raise(tmp_path):
    ds = make_dataset(SynthConfig(dnms_per_trio=2, seed=405, coverage=8.0))
    _, cp, ref = _write_pair(ds.reads, 0, tmp_path, cram_opts=dict(method="raw"))
    raw = open(cp, "rb").read()

    def opened(data, name, reference=ref):
        p = str(tmp_path / name)
        open(p, "wb").write(data)
        os.link(cp + ".crai", p + ".crai") if not os.path.exists(p + ".crai") else None
        f = cramio.CramFile(p, reference)
        _all_records(f)
        return f

    with pytest.raises(ValueError, match=r"not a CRAM file.*offset 0"):
        opened(b"BAM\x01" + raw[4:], "magic.cram")
    with pytest.raises(ValueError, match=r"EOF container.*offset"):
        opened(raw[: len(raw) - 10], "trunc.cram")
    with pytest.raises(ValueError, match=r"EOF container"):
        opened(raw[: len(raw) // 2] + raw[-38:][:20], "cut.cram")
    hdr_crc = bytearray(raw)
    hdr_crc[28] ^= 0x01                                 # inside the file header container's header
    with pytest.raises(ValueError, match=r"CRC32.*container offset 26"):
        opened(bytes(hdr_crc), "crc.cram")
    c0 = int(cramio.CramFile(cp, ref).crai[0, 3])
    blk = bytearray(raw)
    blk[c0 + 60] ^= 0x40                               # inside the first data container's blocks
    with pytest.raises(ValueError, match=r"container offset %d" % c0):
        opened(bytes(blk), "blkcrc.cram")
    # an unknown block method: a raw block relabelled 7, its CRC fixed
    def relabel(path, out):
        d = bytearray(open(path, "rb").read())
        f = cramio.CramFile(path, ref)
        c = f._container(c0)
        b = f._block(c, c.data_off)
        d[c.data_off] = 7
        d[b.data_off + b.size: b.data_off + b.size + 4] = struct.pack("<I", zlib.crc32(bytes(d[c.data_off:b.data_off + b.size])))
        open(out, "wb").write(bytes(d))
    relabel(cp, str(tmp_path / "m.cram"))
    with pytest.raises(ValueError, match=r"unknown block compression method 7.*container offset %d" % c0):
        opened(open(str(tmp_path / "m.cram"), "rb").read(), "method.cram")
    # read names not preserved
    _patch_block(cp, str(tmp_path / "rn.cram"), b"RN\x01AP", lambda d: d.replace(b"RN\x01AP", b"RN\x00AP"))
    with pytest.raises(ValueError, match=r"read names are not preserved.*container offset"):
        opened(open(str(tmp_path / "rn.cram"), "rb").read(), "rn2.cram")
    # an unknown encoding, and GOLOMB
    for codec, msg in ((12, "unknown encoding 12"), (cramio.E_GOLOMB, "GOLOMB")):
        _patch_block(cp, str(tmp_path / "enc.cram"), b"BF\x01\x01", lambda d: d.replace(b"BF\x01\x01", b"BF" + bytes([codec]) + b"\x01", 1))
        with pytest.raises(ValueError, match=msg):
            opened(open(str(tmp_path / "enc.cram"), "rb").read(), "enc%d.cram" % codec)
    # an overrun stream: the slice claims more records than its blocks hold
    f = cramio.CramFile(cp, ref)
    soff = int(f.crai[0, 4])
    c = f._container(c0)
    b = f._block(c, c.data_off + soff)
    d = bytearray(raw)
    sh = bytearray(d[b.data_off:b.data_off + b.size])
    r = cramio._Reader(bytes(sh))
    r.itf8(); r.itf8(); r.itf8()
    p_n = r.p
    n = r.itf8()
    new_n = cramio.itf8(n + 50)
    assert len(new_n) == r.p - p_n
    sh[p_n:r.p] = new_n
    d[b.data_off:b.data_off + b.size] = sh
    d[b.data_off + b.size:b.data_off + b.size + 4] = struct.pack("<I", zlib.crc32(bytes(d[c.data_off + soff:b.data_off + b.size])))
    with pytest.raises(ValueError, match=r"overruns.*container offset %d" % c0):
        opened(bytes(d), "overrun.cram")
    # the reference does not match the slice MD5
    bad_ref = str(tmp_path / "other.fa")
    write_fasta(bad_ref, f.refs, f.ref_lens, seed=99)
    with pytest.raises(ValueError, match=r"MD5.*container offset"):
        opened(raw, "md5.cram", bad_ref)


def test_load_reads_without_pysam_and_routing(clean_modules, tmp_path):
    ds = make_dataset(SMALL[0])
    fakes.install()
    paths, refs, bams = {}, {}, {}
    for k, kid in enumerate(ds.reads.kids):
        bams[kid], paths[kid], refs[kid] = _write_pair(ds.reads, k, tmp_path)
    sys.modules["pysam"] = None
    dc, db = copy.deepcopy(ds.dnms), copy.deepcopy(ds.dnms)
    for d, e in zip(dc, db):
        d["bam"], d["cram_ref"] = paths[d["kid"]], refs[d["kid"]]
        e["bam"] = bams[e["kid"]]
    got = datasource.load_reads(dc, 5000, 151, 1000000)
    want = datasource.load_reads(db, 5000, 151, 1000000)
    _assert_tables_equal(want, got)
    # BAM and CRAM mixed
    mixed = copy.deepcopy(dc)
    first = ds.reads.kids[0]
    for d in mixed:
        if d["kid"] == first:
            d["bam"] = bams[first]
    _assert_tables_equal(want, datasource.load_reads(mixed, 5000, 151, 1000000))
    # a .crai named after the stem
    stem = str(tmp_path / "stem.cram")
    os.link(paths[first], stem)
    os.link(paths[first] + ".crai", str(tmp_path / "stem.crai"))
    assert cramio.is_native_cram(stem, refs[first])
    # CRAM 3.1, an unindexed CRAM and a bgzipped reference still go to pysam
    v31 = str(tmp_path / "v31.cram")
    raw = bytearray(open(paths[first], "rb").read())
    raw[5] = 1
    open(v31, "wb").write(bytes(raw))
    os.link(paths[first] + ".crai", v31 + ".crai")
    unindexed = str(tmp_path / "u.cram")
    os.link(paths[first], unindexed)
    gz_ref = str(tmp_path / "ref.fa.gz")
    open(gz_ref, "wb").write(gzip.compress(open(refs[first], "rb").read()))
    for name, ref in ((v31, refs[first]), (unindexed, refs[first]), (paths[first], gz_ref)):
        dd = copy.deepcopy(ds.dnms)
        for d in dd:
            d["bam"], d["cram_ref"] = name, ref
        with pytest.raises(ImportError):
            datasource.load_reads(dd, 5000, 151, 1000000)


def test_fasta_index_from_fai_equals_scan(tmp_path):
    p = str(tmp_path / "r.fa")
    write_fasta(p, ["a", "b"], [1000, 77], width=50)
    scan = cramio.Fasta(p)
    with open(p + ".fai", "w") as f:
        for n, (ln, off, lb, lw) in scan.index.items():
            f.write("%s\t%d\t%d\t%d\t%d\n" % (n, ln, off, lb, lw))
    fai = cramio.Fasta(p)
    assert fai.index == scan.index
    seq = "".join(open(p).read().split(">a some description\n")[1].split(">")[0].split())
    assert fai.fetch("a", 37, 420) == seq[37:420].encode() and fai.fetch("b", 70, 200) == scan.fetch("b", 70, 200)


def test_cram_structs_match_header(tmp_path):
    prog = tmp_path / "sizes.c"
    body = []
    for st, dt in (("UnfzCramSlice", cramio.SLICE_DTYPE), ("UnfzCramExt", cramio.EXT_DTYPE), ("UnfzCramRef", cramio.REF_DTYPE)):
        body.append('printf("%%zu ", sizeof(%s));' % st)
        body += ['printf("%%zu ", offsetof(%s, %s));' % (st, n) for n in dt.names]
    prog.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){%s return 0;}\n'
                    % (HEADER, "".join(body)))
    exe = tmp_path / "sizes"
    subprocess.run(["gcc", str(prog), "-o", str(exe)], check=True)
    out = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    want = []
    for dt in (cramio.SLICE_DTYPE, cramio.EXT_DTYPE, cramio.REF_DTYPE):
        want += [dt.itemsize] + [dt.fields[n][1] for n in dt.names]
    assert out == want
    for n in ("unfz_rans4x8_decode_host", "unfz_cram_decode_size_host", "unfz_cram_decode_write_host",
              "unfz_cram_decode_size", "unfz_cram_decode_write"):
        assert n in L.SYMBOLS


# ---- a CRAM assembled byte by byte from the specification ------------------------------------------------------------

HTSLIB_EOF = bytes.fromhex("0f000000ffffffff0fe0454f4600000000010005bdd94f0001000606010001000100ee63014b")


def _itf8(v):
    v &= 0xFFFFFFFF
    if v < 0x80:
        return bytes([v])
    if v < 0x4000:
        return bytes([0x80 | (v >> 8), v & 0xFF])
    if v < 0x200000:
        return bytes([0xC0 | (v >> 16), (v >> 8) & 0xFF, v & 0xFF])
    if v < 0x10000000:
        return bytes([0xE0 | (v >> 24), (v >> 16) & 0xFF, (v >> 8) & 0xFF, v & 0xFF])
    return bytes([0xF0 | (v >> 28), (v >> 20) & 0xFF, (v >> 12) & 0xFF, (v >> 4) & 0xFF, v & 0x0F])


def _block(method, ctype, cid, data):
    b = bytes([method, ctype]) + _itf8(cid) + _itf8(len(data)) + _itf8(len(data)) + data
    return b + struct.pack("<I", zlib.crc32(b))


def _container(ref, start, span, n_rec, n_blocks, landmarks, body):
    h = (struct.pack("<i", len(body)) + _itf8(ref) + _itf8(start) + _itf8(span) + _itf8(n_rec) + b"\0\0"
         + _itf8(n_blocks) + _itf8(len(landmarks)) + b"".join(_itf8(x) for x in landmarks))
    return h + struct.pack("<I", zlib.crc32(h)) + body


def test_eof_container_is_htslibs():
    assert cramio.EOF_CONTAINER == HTSLIB_EOF


def test_hand_assembled_file(tmp_path):
    """One container, one slice, three records: S X I D B i (detached mate) / H b N P q Q with a tag / unmapped with RG."""
    import hashlib
    ref = ("ACGTTGCAAC" * 10).encode()
    fa = str(tmp_path / "t.fa")
    open(fa, "wb").write(b">chrT\n" + ref + b"\n")
    S = cramio.SERIES
    cid = {s: i + 1 for i, s in enumerate(S)}
    streams = {}

    def put(s, v, byte=False):
        streams.setdefault(cid[s], bytearray()).extend(bytes([v]) if byte else _itf8(v))

    def arr(s, v):
        streams.setdefault(100 + cid[s], bytearray()).extend(_itf8(len(v)))
        streams.setdefault(cid[s], bytearray()).extend(v)

    def name(v):
        streams.setdefault(cid["RN"], bytearray()).extend(v + b"\0")
    # record 1: mapped at 11, detached mate, qualities stored
    for s, v in (("BF", 0), ("CF", 1 | 2), ("RL", 10), ("AP", 0), ("RG", -1)):      # AP: delta from the slice start
        put(s, v)
    name(b"r1")
    for s, v in (("MF", 1), ("NS", 0), ("NP", 100), ("TS", -50), ("TL", 0), ("FN", 6)):
        put(s, v)
    put("FC", ord("S"), True); put("FP", 1); arr("SC", b"GG")
    put("FC", ord("X"), True); put("FP", 3); put("BS", 0, True)
    put("FC", ord("I"), True); put("FP", 1); arr("IN", b"TT")
    put("FC", ord("D"), True); put("FP", 2); put("DL", 2)
    put("FC", ord("B"), True); put("FP", 0); put("BA", ord("N"), True); put("QS", 5, True)
    put("FC", ord("i"), True); put("FP", 1); put("BA", ord("A"), True)
    put("MQ", 60)
    for q in range(30, 40):
        put("QS", q, True)
    # record 2: reverse strand, no stored qualities, a tag
    for s, v in (("BF", 0x10), ("CF", 0), ("RL", 6), ("AP", 5), ("RG", -1)):
        put(s, v)
    name(b"r2")
    put("TL", 1)
    streams.setdefault(200, bytearray()).extend(_itf8(4))
    streams.setdefault(201, bytearray()).extend(struct.pack("<i", -7))
    put("FN", 6)
    put("FC", ord("H"), True); put("FP", 1); put("HC", 3)
    put("FC", ord("b"), True); put("FP", 0); arr("BB", b"CAT")
    put("FC", ord("N"), True); put("FP", 3); put("RS", 10)
    put("FC", ord("P"), True); put("FP", 0); put("PD", 1)
    put("FC", ord("q"), True); put("FP", 0); arr("QQ", bytes([20, 21]))
    put("FC", ord("Q"), True); put("FP", 2); put("QS", 7, True)
    put("MQ", 20)
    # record 3: unmapped, placed at 16, read group 0
    for s, v in (("BF", 0x4), ("CF", 1), ("RL", 3), ("AP", 0), ("RG", 0)):
        put(s, v)
    name(b"r3")
    put("TL", 0)
    for c in b"ACN":
        put("BA", c, True)
    for q in (10, 11, 12):
        put("QS", q, True)

    def enc(codec, params):
        return _itf8(codec) + _itf8(len(params)) + params
    ext = lambda i: enc(1, _itf8(i))
    ds = []
    for s in S:
        if s == "RN":
            ds.append(b"RN" + enc(5, b"\0" + _itf8(cid[s])))
        elif s in ("SC", "IN", "BB", "QQ"):
            ds.append(s.encode() + enc(4, ext(100 + cid[s]) + ext(cid[s])))
        elif s != "RI":
            ds.append(s.encode() + ext(cid[s]))
    ds_raw = _itf8(len(ds)) + b"".join(ds)
    td = b"\0XYi\0"
    pm = b"RN\x01" + b"AP\x01" + b"RR\x01" + b"SM" + bytes([0x1B] * 5) + b"TD" + _itf8(len(td)) + td
    pm_raw = _itf8(5) + pm
    key = (ord("X") << 16) | (ord("Y") << 8) | ord("i")
    te_raw = _itf8(1) + _itf8(key) + enc(4, ext(200) + ext(201))
    comp = _itf8(len(pm_raw)) + pm_raw + _itf8(len(ds_raw)) + ds_raw + _itf8(len(te_raw)) + te_raw
    ids = sorted(streams)
    blocks = [_block(0, 5, 0, b"")] + [_block(0, 4, i, bytes(streams[i])) for i in ids]
    start, span = 11, 21
    sh = (_itf8(0) + _itf8(start) + _itf8(span) + _itf8(3) + b"\0" + _itf8(len(blocks)) + _itf8(len(ids) + 1) + _itf8(0)
          + b"".join(_itf8(i) for i in ids) + _itf8(-1) + hashlib.md5(ref[start - 1:start - 1 + span]).digest())
    comp_block = _block(0, 1, 0, comp)
    slice_bytes = _block(0, 2, 0, sh) + b"".join(blocks)
    text = b"@SQ\tSN:chrT\tLN:100\n@RG\tID:g1\n"
    hraw = struct.pack("<i", len(text)) + text
    out = b"CRAM\x03\x00" + b"hand".ljust(20, b"\0") + _container(0, 0, 0, 0, 1, [], _block(0, 0, 0, hraw))
    coff = len(out)
    out += _container(0, start, span, 3, 1 + 1 + len(blocks), [len(comp_block)], comp_block + slice_bytes)
    out += HTSLIB_EOF
    path = str(tmp_path / "hand.cram")
    open(path, "wb").write(out)
    open(path + ".crai", "wb").write(gzip.compress(b"0\t%d\t%d\t%d\t%d\t%d\n" % (start, span, coff, len(comp_block),
                                                                                   len(slice_bytes))))
    cf = cramio.CramFile(path, fa)
    assert cf.refs == ["chrT"] and cf.read_groups == ["g1"]
    buf, offs = cf.fetch_union([(0, 0, 100)])
    rec = bamio.parse_records(buf, offs)
    assert bamio._names(buf, offs, rec["l_name"]) == ["r1", "r2", "r3"]
    assert rec["pos"].tolist() == [10, 15, 15] and rec["flag"].tolist() == [0x20, 0x10, 0x4]
    assert rec["mapq"].tolist() == [60, 20, 0] and rec["end"].tolist() == [17, 31, 16]
    assert rec["next_ref_id"].tolist() == [0, -1, -1] and rec["next_pos"].tolist() == [99, -1, -1]
    assert rec["tlen"].tolist() == [-50, 0, 0]
    ops = "MIDNSHP=X"
    cig = []
    for o, r in zip(offs.tolist(), rec):
        c = buf[o + 36 + r["l_name"]: o + 36 + r["l_name"] + 4 * r["n_cigar"]].copy().view("<u4")
        cig.append("".join("%d%s" % (w >> 4, ops[w & 15]) for w in c.tolist()))
    assert cig == ["2S2M2I2D1M1I2M", "3H3M10N1P3M", ""]
    fx = [cramio._bam_fields(buf, o) for o in offs.tolist()]
    assert [f["seq"] for f in fx] == [b"GGAATTNAGC", b"CATACA", b"ACN"]
    assert [list(f["qual"]) for f in fx] == [list(range(30, 40)), [255, 255, 255, 20, 21, 7], [10, 11, 12]]
    assert fx[1]["tags"] == [(key, struct.pack("<i", -7))] and fx[2]["rg"] == "g1" and fx[0]["tags"] == []
