"""GPU: BAM records decoded on the device (bamio.read_regions(engine=...) -> unfz_bam_parse / unfz_bam_emit_*) give
bit for bit the device columns of the same reads decoded on the host and uploaded with Engine.upload_reads, the batch
phaser gives the same records from them, and the command line reads written BAM files without pysam."""
import copy
import sys

import numpy as np
import pytest

from oracle import fakes
from tests.test_bamio_cpu import CASES, modified
from unfazed_b200 import bamio, datasource
from unfazed_b200.schema import READ_HDR, ReadTable, pack_seq
from unfazed_b200.synth import make_dataset

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    from unfazed_b200.engine import Engine
    return Engine(0)


def _regions(ds, margin=6000):
    reg = {}
    for d in ds.dnms:
        chrom = d["chrom"]
        for p in {int(d["start"]), int(d["end"])}:
            reg.setdefault(d["kid"], {}).setdefault(chrom, []).append((p - margin, p + margin))
    return reg


def _write(reads, tmp_path, **opts):
    paths = {}
    for k, kid in enumerate(reads.kids):
        rows = set(np.concatenate([np.arange(reads.blk_off[b], reads.blk_off[b + 1])
                                   for b in range(reads.n_blocks) if reads.blk_kid[b] == k] or [np.zeros(0, np.int64)]).tolist())
        kopts = dict(opts)
        if "extra_tags" in opts:
            kopts["extra_tags"] = {r: v for r, v in opts["extra_tags"].items() if r in rows}
        paths[kid] = str(tmp_path / ("%s.bam" % kid))
        bamio.write_bam(reads, k, paths[kid], **kopts)
    return paths


def _cols(dr):
    t = lambda x: x.cpu().numpy().view(np.uint8)
    return {"hdr": t(dr.hdr), "cigar": t(dr.cigar), "seq2": t(dr.seq2), "lowq": t(dr.lowq), "nmask": t(dr.nmask),
            "start": t(dr.start), "blk_off": t(dr.blk_off)}


def _compare(engine, paths, regions, thresholds=(20, 31)):
    host = bamio.read_regions(paths, regions, head_reads=1000)
    dev = bamio.read_regions(paths, regions, head_reads=1000, engine=engine, min_gt_qual=thresholds[0])
    assert dev.qual is None and dev.n_qual == host.qual.shape[0] and host.n_reads > 0
    assert np.array_equal(dev.hdr, host.hdr) and np.array_equal(dev.cigar, host.cigar) and dev.names == host.names
    for q in thresholds:
        want = _cols(engine.upload_reads(host, min_gt_qual=q))
        got = _cols(dev.device_source.device_reads(q))
        for k in want:
            assert want[k].shape == got[k].shape and np.array_equal(want[k], got[k]), (q, k)
    return host, dev


@pytest.mark.parametrize("cfg", CASES, ids=[str(c.seed) for c in CASES])
def test_device_decode_equals_host_upload(engine, tmp_path, cfg):
    ds = make_dataset(cfg)
    _compare(engine, _write(ds.reads, tmp_path), _regions(ds))


def test_device_decode_tags_iupac_missing_quals(engine, tmp_path):
    ds = make_dataset(CASES[0])
    reads, opts = modified(ds)
    host, _ = _compare(engine, _write(reads, tmp_path, **opts), _regions(ds))
    assert np.any(host.qual & 0x80)


def test_mate_join_kernel_with_forced_hash_collisions(engine, tmp_path):
    """unfz_bam_mate_join against packers._mate_join: with the real name hashes, and with hashes cut to a few bits so
    that groups hold many names -- every collision must be caught by the name comparison and resolved on the host."""
    import zlib
    from unfazed_b200.packers import _mate_join
    ds = make_dataset(CASES[1])
    paths = _write(ds.reads, tmp_path)
    host = bamio.read_regions(paths, _regions(ds))
    dev = bamio.read_regions(paths, _regions(ds), engine=engine)
    assert np.array_equal(dev.hdr["mate"], host.hdr["mate"])
    want = np.full(host.n_reads, -1, dtype=np.int64)
    for b in range(host.n_blocks):
        lo, hi = int(host.blk_off[b]), int(host.blk_off[b + 1])
        m = _mate_join(host.names[lo:hi], host.hdr["flag"][lo:hi].astype(np.int64))
        want[lo:hi] = np.where(m >= 0, m + lo, -1)
    assert np.array_equal(host.hdr["mate"], want) and (want >= 0).sum() > 100
    blk = np.repeat(np.arange(dev.n_blocks, dtype=np.int32), np.diff(dev.blk_off))
    flag = dev.hdr["flag"].astype(np.int32)
    crc = np.array([zlib.crc32(nm.encode()) for nm in dev.names], dtype=np.uint64)
    for bits in (2, 6):
        h = crc & np.uint64((1 << bits) - 1)
        raw = dev.device_source.mate_join(h, blk, flag)
        assert (raw == -2).sum() > 0
        got = bamio.resolve_left_mates(raw.copy(), dev.names, dev.hdr["flag"], dev.blk_off)
        assert np.array_equal(got, want), bits


def _big_table(n_pairs=520_000, n_long=300, seed=9) -> ReadTable:
    """One kid, two contigs, 150 bp pairs (mate 250 bp downstream) plus single reads of 16-24 kb; some N and IUPAC
    bases."""
    rng = np.random.default_rng(seed)
    n = 2 * n_pairs + n_long
    pc = (np.arange(n_pairs) >= n_pairs // 2).astype(np.int32)
    ps = rng.integers(0, 30_000_000, n_pairs).astype(np.int64)
    contig = np.concatenate([pc, pc, rng.integers(0, 2, n_long).astype(np.int32)])
    start = np.concatenate([ps, ps + 250, rng.integers(0, 30_000_000, n_long)]).astype(np.int64)
    L = np.concatenate([np.full(2 * n_pairs, 150), rng.integers(16_500, 24_000, n_long)]).astype(np.int64)
    flag = np.concatenate([np.full(n_pairs, 99), np.full(n_pairs, 147), np.zeros(n_long, np.int64)])
    name = ["p%d" % i for i in range(n_pairs)] * 2 + ["l%d" % i for i in range(n_long)]
    partner = np.concatenate([np.arange(n_pairs) + n_pairs, np.arange(n_pairs), np.full(n_long, -1)])
    order = np.lexsort((start, contig))
    inv = np.empty(n, np.int64)
    inv[order] = np.arange(n)
    contig, L, start, flag, partner = contig[order], L[order], start[order], flag[order], partner[order]
    hdr = np.zeros(n, READ_HDR)
    hdr["start"], hdr["flag"], hdr["mapq"], hdr["l_seq"], hdr["n_cigar"] = start, flag, 60, L, 1
    hdr["tlen"] = np.where(flag == 99, 400, np.where(flag == 147, -400, 0))
    hdr["aux"] = np.where(flag != 0, 1, 0)
    hdr["cigar_off"] = np.arange(n)
    q0 = np.cumsum(L) - L
    hdr["qoff_lo"], hdr["qoff_hi"] = q0 & 0xFFFFFFFF, q0 >> 32
    hdr["mate"] = np.where(partner >= 0, inv[np.maximum(partner, 0)], -1)
    Q = int(L.sum())
    qual = rng.integers(2, 41, Q).astype(np.uint8)
    esc = rng.random(Q) < 0.001
    qual[esc] |= 0x80
    code = rng.integers(0, 4, Q).astype(np.uint8)
    code[esc] = rng.integers(0, 2, int(esc.sum()))
    cig = ((L << 4) | 0).astype(np.uint32)
    bo = np.array([0, int((contig == 0).sum()), n], np.int64)
    return ReadTable(kids=["big"], contigs=["1", "2"], blk_kid=np.zeros(2, np.int32), blk_contig=np.array([0, 1], np.int32),
                     blk_off=bo, hdr=hdr, cigar=cig, qual=qual, seq2=pack_seq(code), names=[name[i] for i in order.tolist()])


def test_device_decode_one_million_reads_with_long_reads(engine, tmp_path):
    t = _big_table()
    path = str(tmp_path / "big.bam")
    bamio.write_bam(t, 0, path, level=1)
    regions = {"big": {"1": [(0, 40_000_000)], "2": [(0, 40_000_000)]}}
    host, dev = _compare(engine, {"big": path}, regions)
    assert host.n_reads >= 1_000_000 and int(host.hdr["l_seq"].max()) > 16 * 1024


def test_batch_phaser_records_from_device_decoded_reads(engine, tmp_path):
    from unfazed_b200.phaser import BatchPhaser
    ds = make_dataset(CASES[1])
    paths = _write(ds.reads, tmp_path)
    dnms = copy.deepcopy(ds.dnms)
    for d in dnms:
        d["bam"] = paths[d["kid"]]
    host = datasource.load_reads(dnms, 5000, 151, 1000000)
    dev = datasource.load_reads(dnms, 5000, 151, 1000000, engine=engine, min_gt_qual=20)
    want = BatchPhaser(engine, ds.sites, host, ds.pedigrees).phase(copy.deepcopy(ds.dnms), threads=1)
    bp = BatchPhaser(engine, ds.sites, dev, ds.pedigrees, dreads=dev.device_reads)
    got = bp.phase(copy.deepcopy(ds.dnms), threads=1)
    assert set(got) == set(want) and len(want) > 0
    for k in want:
        assert got[k] == want[k], k
    # another --min-gt-qual: the planes are emitted again from the resident records
    want2 = BatchPhaser(engine, ds.sites, host, ds.pedigrees).phase(copy.deepcopy(ds.dnms), threads=1, min_gt_qual=35)
    got2 = bp.phase(copy.deepcopy(ds.dnms), threads=1, min_gt_qual=35)
    assert bp.dreads.min_bq == 35 and got2 == want2


@pytest.mark.parametrize("name", ["snv_noisy", "indel_cluster_many", "sv_cnv", "sexchrom_chr", "no_extended"])
def test_cli_bed_from_written_bam_without_pysam(engine, tmp_path, name):
    from oracle.make_golden import cli_files
    from tests.golden_util import load_case
    from tests.test_gpu_golden import _bed_rows
    from unfazed_b200.__main__ import main
    ds, want = load_case(name)
    bed, ped, pairs = cli_files(ds, str(tmp_path))
    vcf_name = "mem://golden.vcf"
    datasource._registry.clear()
    fakes.install()
    fakes.register_vcf(vcf_name, ds.sites)
    saved = sys.modules.get("pysam")
    sys.modules["pysam"] = None                       # BAM input must not need pysam
    try:
        for kid, path in pairs:
            bamio.write_bam(ds.reads, ds.reads.kids.index(kid), path)
        p = dict(threads=1, build="38", multiread_proc_min=1000, no_extended=False)
        p.update(ds.params)
        for amb in (False, True):
            out = tmp_path / ("out_%s.bed" % amb)
            argv = ["-d", bed, "-s", vcf_name, "-p", ped, "--bam-pairs"] + ["%s:%s" % (k, b) for k, b in pairs] + \
                   ["-t", str(p["threads"]), "-g", p["build"], "--multiread-proc-min", str(p["multiread_proc_min"]),
                    "--quiet", "--verbose", "-o", "bed", "--outfile", str(out)]
            if p["no_extended"]:
                argv.append("--no-extended")
            if amb:
                argv.append("--include-ambiguous")
            main(argv)
            assert _bed_rows(out.read_text()) == _bed_rows(want["cli"]["ambiguous" if amb else "strict"]), (name, amb)
    finally:
        if saved is None:
            sys.modules.pop("pysam", None)
        else:
            sys.modules["pysam"] = saved
        if getattr(sys.modules.get("cyvcf2"), "__fake__", False):
            del sys.modules["cyvcf2"]
        datasource._registry.clear()
