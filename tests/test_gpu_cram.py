"""GPU: CRAM slices decoded on the device (cram_slice_size_kernel / cram_slice_write_kernel) give the host decode's
records byte for byte, the same DeviceReads and batch-phaser records as the BAM of the same reads, and the command line
reads CRAMs plus a FASTA without pysam."""
import copy
import sys

import numpy as np
import pytest

from oracle import fakes
from tests.test_cramio_cpu import SMALL, _all_records, _regions, _write_pair, noisy, write_fasta
from tests.test_gpu_bam import _big_table, _cols
from unfazed_b200 import bamio, cramio, datasource
from unfazed_b200.synth import make_dataset

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    from unfazed_b200.engine import Engine
    return Engine(0)


def _device_equals_host(engine, cp, ref):
    host = cramio.CramFile(cp, ref)
    dev = cramio.CramFile(cp, ref, engine=engine)
    hb, ho = _all_records(host)
    db, do = _all_records(dev)
    assert hb.tobytes() == db.tobytes() and np.array_equal(ho, do) and ho.shape[0] > 0
    assert bytes(db.resident[: db.shape[0]].cpu().numpy()) == hb.tobytes()
    return ho.shape[0]


def test_device_decode_equals_host_decode(engine, tmp_path):
    ds = make_dataset(SMALL[0])
    reads, opts = noisy(ds)
    variants = [dict(), dict(method="raw", encoding="core"), dict(method="lzma", multi_ref=True, records_per_slice=2000),
                dict(method="rans1", rr=False), dict(method="bzip2", embed_ref=True, records_per_slice=200)]
    rows = set(np.concatenate([np.arange(reads.blk_off[b], reads.blk_off[b + 1]) for b in range(reads.n_blocks)
                               if reads.blk_kid[b] == 0]).tolist())
    opts["extra_tags"] = {r: v for r, v in opts["extra_tags"].items() if r in rows}
    for i, v in enumerate(variants):
        _, cp, ref = _write_pair(reads, 0, tmp_path, cram_opts=v, bam_opts=opts, tag="g%d" % i)
        _device_equals_host(engine, cp, ref)


def test_device_decode_many_reads_with_long_reads(engine, tmp_path):
    t = _big_table(n_pairs=30_000, n_long=30)
    bp = str(tmp_path / "big.bam")
    bamio.write_bam(t, 0, bp, level=1)
    f = bamio.BamFile(bp)
    ref = str(tmp_path / "big.fa")
    write_fasta(ref, f.refs, f.ref_lens)
    cp = str(tmp_path / "big.cram")
    cramio.write_cram(t, 0, cp, ref, method="gzip", records_per_slice=4000)
    n = _device_equals_host(engine, cp, ref)
    assert n == t.n_reads and int(t.hdr["l_seq"].max()) > 16 * 1024


def _load(dnms, paths, refs, engine=None, q=20):
    dd = copy.deepcopy(dnms)
    for d in dd:
        d["bam"] = paths[d["kid"]]
        d["cram_ref"] = refs.get(d["kid"]) if refs else None
    return datasource.load_reads(dd, 5000, 151, 1000000, engine=engine, min_gt_qual=q)


def test_device_reads_and_phaser_records_from_cram_equal_bam(engine, tmp_path):
    from unfazed_b200.phaser import BatchPhaser
    ds = make_dataset(SMALL[1])
    bams, crams, refs = {}, {}, {}
    for k, kid in enumerate(ds.reads.kids):
        bams[kid], crams[kid], refs[kid] = _write_pair(ds.reads, k, tmp_path, cram_opts=dict(records_per_slice=500))
    want = _load(ds.dnms, bams, None, engine)
    got = _load(ds.dnms, crams, refs, engine)
    assert np.array_equal(got.hdr, want.hdr) and np.array_equal(got.cigar, want.cigar) and got.names == want.names
    for q in (20, 31):
        a = _cols(want.device_source.device_reads(q))
        b = _cols(got.device_source.device_reads(q))
        for key in a:
            assert np.array_equal(a[key], b[key]), (q, key)
    host = _load(ds.dnms, bams, None)
    rec_want = BatchPhaser(engine, ds.sites, host, ds.pedigrees).phase(copy.deepcopy(ds.dnms), threads=1)
    bp = BatchPhaser(engine, ds.sites, got, ds.pedigrees, dreads=got.device_source.device_reads(20))
    rec_got = bp.phase(copy.deepcopy(ds.dnms), threads=1)
    assert rec_got == rec_want and len(rec_want) > 0
    st = engine.cram_decoder()
    assert st.h2d_bytes > 0 and {"size", "write"} <= set(st.timings_ms)


@pytest.mark.parametrize("name", ["snv_noisy", "indel_cluster_many", "sv_cnv", "sexchrom_chr", "no_extended"])
def test_cli_bed_from_written_cram_without_pysam(engine, tmp_path, name):
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
    sys.modules["pysam"] = None                       # CRAM input must not need pysam
    try:
        ref = str(tmp_path / "ref.fa")
        write_fasta(ref, ds.reads.contigs, [int(ds.reads.ref_ends().max()) + 1000] * len(ds.reads.contigs))
        cram_pairs = []
        for kid, path in pairs:
            k = ds.reads.kids.index(kid)
            cp = path[:-4] + ".cram"
            cramio.write_cram(ds.reads, k, cp, ref)
            cram_pairs.append((kid, cp))
        p = dict(threads=1, build="38", multiread_proc_min=1000, no_extended=False)
        p.update(ds.params)
        for amb in (False, True):
            out = tmp_path / ("out_%s.bed" % amb)
            argv = ["-d", bed, "-s", vcf_name, "-p", ped, "-r", ref, "--bam-pairs"] + \
                   ["%s:%s" % (k, b) for k, b in cram_pairs] + \
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
