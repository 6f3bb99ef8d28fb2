"""CPU: the native BAM reader (bamio) -- BGZF, header, BAI queries, and the ReadTable it builds, which must equal what
packers.pack_reads builds from the pysam API (here the in-memory fakes) over the same reads, array for array."""
import copy
import ctypes
import gzip
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import fakes
from unfazed_b200 import _lib as L
from unfazed_b200 import bamio, datasource
from unfazed_b200.schema import AUX_HAS_SA, AUX_SAME_REF, QUAL_ESCAPE, pack_seq
from unfazed_b200.synth import SynthConfig, make_dataset

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "unfazed_sm100.h")

CASES = [
    SynthConfig(dnms_per_trio=8, seed=301, coverage=20.0),
    SynthConfig(dnms_per_trio=6, seed=302, coverage=20.0, n_trios=2, sv_frac=0.4, sv_max_len=20000, indel_frac=0.2),
    SynthConfig(dnms_per_trio=6, seed=303, coverage=20.0, chr_prefix="chr", sex_chrom_frac=0.3, male_frac=1.0),
]


@pytest.fixture(scope="module", autouse=True)
def native_lib():
    if not os.path.exists(L.LIB_PATH):
        import __graft_entry__ as g
        g.build()


@pytest.fixture()
def fake_decoders():
    fakes.install()
    datasource._registry.clear()
    yield
    datasource._registry.clear()
    for m in ("cyvcf2", "pysam"):
        if m in sys.modules and (sys.modules[m] is None or getattr(sys.modules[m], "__fake__", False)):
            del sys.modules[m]


def modified(ds, seed=11):
    """The dataset's reads with SA and other tags, mates on another contig, IUPAC / '=' bases and missing qualities:
    the table to compare on and the writer's options that put those features into the file."""
    rng = np.random.default_rng(seed)
    t = copy.deepcopy(ds.reads)
    n = t.n_reads
    t.names = t.names_of(np.arange(n))               # pair names stay what they were when mate pointers change
    sa = rng.random(n) < 0.1
    t.hdr["aux"] = t.hdr["aux"] | np.where(sa, AUX_HAS_SA, 0).astype(np.uint8)
    # mates on another reference: next_refID differs, so neither the packer nor the reader resolves them
    other = np.flatnonzero((rng.random(n) < 0.05) & ((t.hdr["aux"] & AUX_SAME_REF) != 0))
    t.hdr["aux"][other] &= ~np.uint8(AUX_SAME_REF)
    t.hdr["mate"][other] = -1
    # escaped bases: N (code 0) and other IUPAC letters or '=' (code 1)
    Q = t.qual.shape[0]
    g = np.arange(Q)
    code = ((t.seq2[g >> 2] >> ((g & 3) << 1).astype(np.uint8)) & 3).astype(np.uint8)
    esc = np.flatnonzero(rng.random(Q) < 0.002)
    code[esc] = rng.integers(0, 2, esc.shape[0])
    t.qual[esc] |= QUAL_ESCAPE
    t.seq2 = pack_seq(code)
    # missing quality strings: every quality 0 (the escape bits stay)
    missing = np.flatnonzero((rng.random(n) < 0.03) & (t.hdr["l_seq"] > 0))
    for r in missing.tolist():
        q0 = t.qoff(r)
        t.qual[q0:q0 + int(t.hdr["l_seq"][r])] &= QUAL_ESCAPE
    tags = {}
    for r in np.flatnonzero(rng.random(n) < 0.2).tolist():
        tags[r] = (bamio.encode_tag("NM", "i", int(r % 7)) + bamio.encode_tag("RG", "Z", "SAmple1")
                   + bamio.encode_tag("XB", "B", ("s", [1, -2, 3])) + bamio.encode_tag("XF", "f", 0.5)
                   + bamio.encode_tag("XA", "A", "S") + bamio.encode_tag("XC", "c", -3) + bamio.encode_tag("XS", "S", 513)
                   + bamio.encode_tag("XH", "H", "53410A") + bamio.encode_tag("XI", "I", 7))
    return t, dict(extra_tags=tags, missing_qual=missing, other_ref=other)


def _write_all(reads, tmp_path, **opts):
    paths = {}
    for k, kid in enumerate(reads.kids):
        p = str(tmp_path / ("%s.bam" % kid))
        kopts = dict(opts)
        if opts:
            rows = set(np.flatnonzero(np.isin(np.arange(reads.n_reads), np.concatenate(
                [np.arange(reads.blk_off[b], reads.blk_off[b + 1]) for b in range(reads.n_blocks) if reads.blk_kid[b] == k]
                or [np.zeros(0, np.int64)]))).tolist())
            kopts["extra_tags"] = {r: v for r, v in opts["extra_tags"].items() if r in rows}
        bamio.write_bam(reads, k, p, **kopts)
        paths[kid] = p
    return paths


def _both(ds, reads, paths):
    """(packer over the fakes, bamio) through datasource.load_reads, for the DNMs of the dataset."""
    dm, db = copy.deepcopy(ds.dnms), copy.deepcopy(ds.dnms)
    for d, e in zip(dm, db):
        d["bam"], d["cram_ref"] = "mem://%s.bam" % d["kid"], None
        fakes.register_bam(d["bam"], reads, reads.kids.index(d["kid"]))
        e["bam"] = paths[e["kid"]]
    want = datasource.load_reads(dm, 5000, 151, 1000000)
    got = datasource.load_reads(db, 5000, 151, 1000000)
    return want, got


def _assert_tables_equal(want, got):
    assert list(got.kids) == list(want.kids) and list(got.contigs) == list(want.contigs)
    for f in ("blk_kid", "blk_contig", "blk_off", "hdr", "cigar", "qual", "seq2"):
        a, b = getattr(want, f), getattr(got, f)
        assert a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a, b), f
    assert got.names == want.names
    assert set(got.head_tlen) == set(want.head_tlen)
    for k in want.head_tlen:
        assert np.array_equal(got.head_tlen[k], want.head_tlen[k]), k


@pytest.mark.parametrize("cfg", CASES, ids=[str(c.seed) for c in CASES])
def test_read_regions_equals_packer(fake_decoders, tmp_path, cfg):
    ds = make_dataset(cfg)
    paths = _write_all(ds.reads, tmp_path)
    want, got = _both(ds, ds.reads, paths)
    assert want.n_reads > 0
    _assert_tables_equal(want, got)


def test_read_regions_equals_packer_tags_iupac_missing_quals(fake_decoders, tmp_path):
    ds = make_dataset(CASES[0])
    reads, opts = modified(ds)
    paths = _write_all(reads, tmp_path, **opts)
    want, got = _both(ds, reads, paths)
    _assert_tables_equal(want, got)
    assert np.any(got.hdr["aux"] & AUX_HAS_SA) and np.any(got.qual & QUAL_ESCAPE)


def _records_of(path):
    """Every record of a BAM by a sequential walk (brute force, no index): (bytes, offsets, parsed fields)."""
    f = bamio.BamFile(path)
    buf, _ = f.bgzf.stream_from(f.first_voff, 1 << 40)
    offs, end = bamio.record_offsets(buf)
    assert end == buf.shape[0]
    return f, buf, offs, bamio.parse_records(buf, offs)


def test_round_trip_bytes_header_and_records(tmp_path):
    ds = make_dataset(CASES[0])
    t = copy.deepcopy(ds.reads)
    t.contigs = list(t.contigs) + ["empty_contig"]
    path = str(tmp_path / "k.bam")
    bamio.write_bam(t, 0, path)
    raw = open(path, "rb").read()
    assert raw.endswith(bamio.BGZF_EOF)
    # every BGZF member inflates with the standard gzip reader to the same bytes bamio reads
    plain = gzip.decompress(raw)
    f, buf, offs, rec = _records_of(path)
    assert plain[f.header_bytes:] == buf.tobytes()
    assert f.refs == list(t.contigs) and len(f.ref_lens) == len(t.contigs)
    # records straddle block boundaries
    starts = offs + f.header_bytes
    ends = starts + 4 + buf[offs[:, None] + np.arange(4)].copy().view("<i4").reshape(-1)
    assert np.any(starts // 0xFF00 != (ends - 1) // 0xFF00)
    # field for field against the table
    rows = np.concatenate([np.arange(t.blk_off[b], t.blk_off[b + 1]) for b in range(t.n_blocks) if t.blk_kid[b] == 0])
    h = t.hdr[rows]
    assert np.array_equal(rec["pos"], h["start"]) and np.array_equal(rec["flag"], h["flag"])
    assert np.array_equal(rec["tlen"], h["tlen"]) and np.array_equal(rec["mapq"], h["mapq"])
    assert np.array_equal(rec["l_seq"], h["l_seq"]) and np.array_equal(rec["n_cigar"], h["n_cigar"])
    assert np.array_equal(rec["pos"].astype(np.int64) + rec["ref_len"], t.ref_ends()[rows])
    names = bamio._names(buf, offs, rec["l_name"])
    assert names == t.names_of(rows)
    cig = bamio.gather(buf, offs + 36 + rec["l_name"], 4 * rec["n_cigar"].astype(np.int64)).view("<u4")
    assert np.array_equal(cig, t.cigar[np.concatenate([np.arange(o, o + n) for o, n in zip(h["cigar_off"], h["n_cigar"])])])
    # the empty reference answers with nothing
    assert f.query("empty_contig", 0, 1000)[1].shape[0] == 0


def test_corrupt_and_truncated_files_raise(tmp_path):
    ds = make_dataset(SynthConfig(dnms_per_trio=3, seed=305, coverage=10.0))
    path = str(tmp_path / "k.bam")
    bamio.write_bam(ds.reads, 0, path)
    raw = bytearray(open(path, "rb").read())
    trunc = tmp_path / "trunc.bam"
    trunc.write_bytes(bytes(raw[: len(raw) // 2]))
    with pytest.raises(ValueError, match="EOF"):
        bamio.BgzfReader(str(trunc))
    # a truncated block before an intact EOF marker
    cut = tmp_path / "cut.bam"
    cut.write_bytes(bytes(raw[: len(raw) // 2]) + bamio.BGZF_EOF)
    r = bamio.BgzfReader(str(cut))
    with pytest.raises(ValueError):
        c = 0
        while True:
            c += r.block_size(c)
    # a wrong stored CRC32 (the first of the last 8 bytes of the first block): the data inflate, the check fails
    size0 = bamio.BgzfReader(path).block_size(0)
    bad = bytearray(raw)
    bad[size0 - 8] ^= 0xFF
    p2 = tmp_path / "crc.bam"
    p2.write_bytes(bytes(bad))
    with pytest.raises(ValueError, match="CRC32"):
        bamio.BgzfReader(str(p2)).inflate([0])
    # a wrong ISIZE
    bad = bytearray(raw)
    bad[size0 - 1] ^= 0x01
    p3 = tmp_path / "isize.bam"
    p3.write_bytes(bytes(bad))
    with pytest.raises(ValueError, match="ISIZE"):
        bamio.BgzfReader(str(p3)).inflate([0])


def test_bai_queries_equal_brute_force_scan(tmp_path):
    ds = make_dataset(CASES[1])
    t = ds.reads
    path = str(tmp_path / "k.bam")
    bamio.write_bam(t, 0, path)
    f, buf, offs, rec = _records_of(path)
    rng = np.random.default_rng(5)
    n_checked = 0
    for it in range(300):
        tid = int(rng.integers(0, len(f.refs)))
        ln = f.ref_lens[tid]
        kind = it % 5
        if kind == 0:
            beg = end = int(rng.integers(0, ln))                      # zero-length
        elif kind == 1:
            beg, end = max(0, ln - int(rng.integers(1, 3000))), ln    # contig end
        elif kind == 2:
            beg, end = 0, int(rng.integers(1, 5000))                  # contig start
        else:
            beg = int(rng.integers(0, ln))
            end = beg + int(rng.integers(1, 40000))
        _, qo, qr = f.query(f.refs[tid], beg, end)
        want = np.flatnonzero((rec["ref_id"] == tid) & (rec["pos"] < end) & (rec["end"] > beg))
        got_bytes = [buf.tobytes()[o: o + 36] for o in offs[want]]
        assert qr.shape[0] == want.shape[0], (tid, beg, end)
        assert np.array_equal(qr, rec[want])
        qb, qo2, _ = f.query(f.refs[tid], beg, end)
        assert [qb.tobytes()[o: o + 36] for o in qo2] == got_bytes
        n_checked += want.shape[0]
    assert n_checked > 0
    with pytest.raises(ValueError):
        f.query("no_such_contig", 0, 10)


def test_load_reads_without_pysam_and_routing(fake_decoders, tmp_path):
    ds = make_dataset(CASES[0])
    paths = _write_all(ds.reads, tmp_path)
    want, _ = _both(ds, ds.reads, paths)
    sys.modules["pysam"] = None                       # import pysam now raises ImportError
    db = copy.deepcopy(ds.dnms)
    for d in db:
        d["bam"] = paths[d["kid"]]
    got = datasource.load_reads(db, 5000, 151, 1000000)
    _assert_tables_equal(want, got)
    # CRAM, an unindexed BAM and registered mem:// names still go to pysam
    cram = str(tmp_path / "x.cram")
    open(cram, "wb").close()
    unindexed = str(tmp_path / "u.bam")
    bamio.write_bam(ds.reads, 0, unindexed)
    os.remove(unindexed + ".bai")
    for name in (cram, unindexed, "mem://x.bam"):
        dd = copy.deepcopy(ds.dnms)
        for d in dd:
            d["bam"] = name
        with pytest.raises(ImportError):
            datasource.load_reads(dd, 5000, 151, 1000000)


def test_device_decoded_table_refuses_host_planes(tmp_path):
    from unfazed_b200.engine import PackedReads
    ds = make_dataset(SynthConfig(dnms_per_trio=3, seed=306, coverage=10.0))
    t = copy.deepcopy(ds.reads)
    t.n_bases, t.qual, t.seq2 = int(t.qual.shape[0]), None, None
    t.validate()
    assert t.n_qual == int(ds.reads.qual.shape[0])
    with pytest.raises(ValueError, match="decoded on the device"):
        PackedReads(t, 20)
    with pytest.raises(ValueError, match="decoded on the device"):
        t.lowq_plane(20)


def test_bam_record_struct_matches_header(tmp_path):
    prog = tmp_path / "sizes.c"
    fields = [n for n in L.BAM_REC_DTYPE.names]
    prog.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){printf("%%zu", sizeof(UnfzBamRec));%s'
                    'return 0;}\n' % (HEADER, "".join('printf(" %%zu", offsetof(UnfzBamRec, %s));' % n for n in fields)))
    exe = tmp_path / "sizes"
    subprocess.run(["gcc", str(prog), "-o", str(exe)], check=True)
    out = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert out[0] == L.BAM_REC_DTYPE.itemsize == 48
    assert out[1:] == [L.BAM_REC_DTYPE.fields[n][1] for n in fields]
    lib = ctypes.CDLL(L.LIB_PATH)
    for n in ("unfz_bam_record_offsets", "unfz_bam_parse_host", "unfz_bam_gather_host", "unfz_bam_parse",
              "unfz_bam_emit_cigar", "unfz_bam_emit_planes"):
        assert hasattr(lib, n) and n in L.SYMBOLS
