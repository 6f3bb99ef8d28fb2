"""GPU: VCF text decoded on the device (vcfio.read_sites(engine=...) -> unfz_vcf_line_count / unfz_vcf_line_write /
unfz_vcf_parse / unfz_vcf_samples) gives bit for bit the table of the host decode, the batch phaser gives the same
records from it, and the command line reads a written sites VCF and BAMs with neither cyvcf2 nor pysam."""
import copy
import gzip
import sys

import numpy as np
import pytest

from oracle import fakes
from tests.golden_util import CASES as GOLDEN_CASES, load_case
from tests.test_vcfio_cpu import assert_tables_equal, dnm_regions, write_text_vcf
from unfazed_b200 import bamio, datasource, packers, vcfio

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    from unfazed_b200.engine import Engine
    return Engine(0)


def _device_equals_host(engine, path, trios, regions, max_digits=15):
    host = vcfio.read_sites(path, trios, regions, max_digits=max_digits)
    dev = vcfio.read_sites(path, trios, regions, engine=engine, max_digits=max_digits)
    assert_tables_equal(host, dev)
    assert np.array_equal(host.gq.view(np.uint32), dev.gq.view(np.uint32))
    # the fixed fields of every line of the inflated chunks, bit for bit
    vf = vcfio.VcfFile(path)
    qs = [(vf.tids[c], max(a, 0), max(b, 1)) for c, ivs in regions.items() if c in vf.tids for a, b in vcfio._merge(ivs)]
    buf, _ = vf.fetch_union(qs)
    want = vcfio.HostDecoder().lines(buf)
    got = engine.vcf_decoder().lines(buf)
    assert want.shape[0] > 0 and np.array_equal(want.view(np.uint8), got.view(np.uint8))
    return host, dev


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_device_equals_host_golden(engine, tmp_path, name):
    ds, _ = load_case(name)
    path = str(tmp_path / "g.vcf.gz")
    vcfio.write_vcf(ds.sites, path)
    prefix = "chr" if ds.sites.contigs[0].startswith("chr") else ""
    host, _ = _device_equals_host(engine, path, ds.sites.trios, dnm_regions(ds.dnms, prefix))
    fakes.register_vcf("mem://g", ds.sites)
    assert_tables_equal(packers.pack_sites(fakes.VCF("mem://g"), ds.sites.trios, dnm_regions(ds.dnms, prefix)), host)


def _random_lines(rng, n_samples, n_lines, float_gq):
    """Lines with a random FORMAT layout per line (GT GQ AD RO AO DP PL, any order, some absent), missing values,
    dropped trailing fields, phased / haploid / multi-allelic genotypes."""
    keys = ["GT", "GQ", "AD", "RO", "AO", "DP", "PL"]
    lines, pos = [], 100
    for _ in range(n_lines):
        pos += int(rng.integers(1, 400))
        fmt = [k for k in keys if rng.random() < 0.8] or ["GT"]
        rng.shuffle(fmt)
        n_alt = int(rng.integers(1, 3))
        cells = []
        for _s in range(n_samples):
            v = []
            for k in fmt:
                r = rng.random()
                if k == "GT":
                    al = lambda: "." if rng.random() < 0.1 else str(int(rng.integers(0, n_alt + 1)))
                    v.append(al() if r < 0.05 else al() + ("|" if rng.random() < 0.3 else "/") + al())
                elif k == "GQ":
                    x = rng.uniform(0, 99)
                    v.append("." if r < 0.1 else ("%.*f" % (int(rng.integers(0, 9)), x) if float_gq else str(int(x))))
                elif k in ("AD", "AO", "PL"):
                    m = n_alt + 1 if k != "AO" else n_alt
                    v.append("." if r < 0.1 else ",".join("." if rng.random() < 0.05 else str(int(rng.integers(0, 300)))
                                                          for _ in range(m)))
                else:
                    v.append("." if r < 0.1 else str(int(rng.integers(0, 500))))
            while len(v) > 1 and rng.random() < 0.1:
                v.pop()                                           # dropped trailing fields
            cells.append(":".join(v))
        alt = ",".join("ACGT"[int(rng.integers(0, 4))] for _ in range(n_alt))
        lines.append("\t".join(["1", str(pos), ".", "A", alt, ".", ".", "DP=1", ":".join(fmt)] + cells))
    return lines


@pytest.mark.parametrize("float_gq", [False, True])
def test_device_equals_host_random_layouts(engine, tmp_path, float_gq):
    rng = np.random.default_rng(11 + float_gq)
    samples = ["s%d" % i for i in range(30)]
    lines = _random_lines(rng, 30, 400, float_gq)
    path = write_text_vcf(tmp_path, samples, lines, "Float" if float_gq else "Integer")
    trios = [tuple(samples[i: i + 3]) for i in range(0, 27, 3)]              # s27..s29 are not members
    host, _ = _device_equals_host(engine, path, trios, {"1": [(0, 10 ** 6)]})
    assert host.n_rows == 400 * len(trios)


def test_device_equals_host_1000_trio_lines_over_64kb(engine, tmp_path):
    rng = np.random.default_rng(5)
    samples = ["s%d" % i for i in range(3000)]
    lines = _random_lines(rng, 3000, 24, True)
    assert max(len(l) for l in lines) > 64 * 1024
    path = write_text_vcf(tmp_path, samples, lines, "Float")
    trios = [tuple(samples[i: i + 3]) for i in range(0, 3000, 3)]
    _device_equals_host(engine, path, trios, {"1": [(0, 10 ** 6)]})


def test_floats_forced_off_the_fast_path(engine, tmp_path):
    """With max_digits=0 every float GQ goes to the host decode; the fast path must give the same bits."""
    rng = np.random.default_rng(8)
    samples = ["s%d" % i for i in range(60)]
    lines = _random_lines(rng, 60, 100, True)
    path = write_text_vcf(tmp_path, samples, lines, "Float")
    trios = [tuple(samples[i: i + 3]) for i in range(0, 60, 3)]
    fast, _ = _device_equals_host(engine, path, trios, {"1": [(0, 10 ** 6)]})
    slow, _ = _device_equals_host(engine, path, trios, {"1": [(0, 10 ** 6)]}, max_digits=0)
    assert_tables_equal(fast, slow)
    assert np.array_equal(fast.gq.view(np.uint32), slow.gq.view(np.uint32))
    assert np.any(fast.gq != np.round(fast.gq))


def test_batch_phaser_records_from_device_decoded_sites(engine, tmp_path):
    from tests.test_bamio_cpu import CASES
    from unfazed_b200.phaser import BatchPhaser
    from unfazed_b200.synth import make_dataset
    ds = make_dataset(CASES[1])
    path = str(tmp_path / "b.vcf.gz")
    vcfio.write_vcf(ds.sites, path)
    datasource._registry.clear()
    dev = datasource.load_sites(path, ds.dnms, ds.pedigrees, 5000, engine=engine)
    want = BatchPhaser(engine, ds.sites, ds.reads, ds.pedigrees).phase(copy.deepcopy(ds.dnms), threads=1)
    got = BatchPhaser(engine, dev, ds.reads, ds.pedigrees).phase(copy.deepcopy(ds.dnms), threads=1)
    assert set(got) == set(want) and len(want) > 0
    for k in want:
        assert got[k] == want[k], k


def _dnm_vcf(ds, path):
    kids = sorted({d["kid"] for d in ds.dnms})
    lines = []
    for d in ds.dnms:
        sv = d["vartype"] in ("DEL", "DUP", "INV", "CNV", "DUP:TANDEM", "DEL:ME", "CPX", "CTX")
        ref = "N" if sv else "N" * max(int(d["end"]) - int(d["start"]), 1)
        info = "SVTYPE=%s;END=%d" % (d["vartype"], int(d["end"])) if sv else "."
        gts = ["0/1" if k == d["kid"] else "0/0" for k in kids]
        lines.append("\t".join([d["chrom"], str(int(d["start"]) + 1), ".", ref, "<%s>" % d["vartype"] if sv else "A",
                                ".", ".", info, "GT"] + gts))
    with gzip.open(path, "wt") as f:
        f.write("##fileformat=VCFv4.2\n" + "\t".join(["#CHROM", "POS", "ID", "REF", "ALT", "QUAL", "FILTER", "INFO",
                                                     "FORMAT"] + kids) + "\n" + "\n".join(lines) + "\n")


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_cli_bed_from_written_vcf_and_bams_without_cyvcf2_or_pysam(engine, tmp_path, name):
    from oracle.make_golden import cli_files
    from tests.test_gpu_golden import _bed_rows
    from unfazed_b200.__main__ import main
    ds, want = load_case(name)
    bed, ped, pairs = cli_files(ds, str(tmp_path))
    sites = str(tmp_path / "sites.vcf.gz")
    vcfio.write_vcf(ds.sites, sites)
    dnm_inputs = [bed]
    if name == "sv_cnv":
        dnm_inputs.append(str(tmp_path / "dnms.vcf.gz"))
        _dnm_vcf(ds, dnm_inputs[-1])
    datasource._registry.clear()
    saved = {m: sys.modules.get(m) for m in ("cyvcf2", "pysam")}
    sys.modules["cyvcf2"] = None                      # neither decoder may be needed
    sys.modules["pysam"] = None
    try:
        for kid, path in pairs:
            bamio.write_bam(ds.reads, ds.reads.kids.index(kid), path)
        p = dict(threads=1, build="38", multiread_proc_min=1000, no_extended=False)
        p.update(ds.params)
        for dnms in dnm_inputs:
            for amb in (False, True):
                out = tmp_path / ("out_%s.bed" % amb)
                argv = ["-d", dnms, "-s", sites, "-p", ped, "--bam-pairs"] + ["%s:%s" % (k, b) for k, b in pairs] + \
                       ["-t", str(p["threads"]), "-g", p["build"], "--multiread-proc-min", str(p["multiread_proc_min"]),
                        "--quiet", "--verbose", "-o", "bed", "--outfile", str(out)]
                if p["no_extended"]:
                    argv.append("--no-extended")
                if amb:
                    argv.append("--include-ambiguous")
                main(argv)
                assert _bed_rows(out.read_text()) == _bed_rows(want["cli"]["ambiguous" if amb else "strict"]), \
                    (name, dnms, amb)
    finally:
        for m, v in saved.items():
            if v is None:
                sys.modules.pop(m, None)
            else:
                sys.modules[m] = v
        datasource._registry.clear()
