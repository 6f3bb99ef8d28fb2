"""GPU: BCF records decoded on the device (bcfio.read_sites(engine=...) -> unfz_bcf_parse / unfz_bcf_samples) give bit
for bit the table of the host decode, the batch phaser gives the same records from it, and the command line reads a
written sites BCF and CSI-indexed BAMs with neither cyvcf2 nor pysam."""
import copy
import sys

import numpy as np
import pytest

from tests.golden_util import CASES as GOLDEN_CASES, load_case
from tests.test_bcfio_cpu import (FEOV, FLOAT, FMISS, HEAD_PLAIN, INT8, INT16, INT32, KEYS, dnm_bcf, record,
                                  write_hand_bcf)
from tests.test_vcfio_cpu import assert_tables_equal, dnm_regions
from unfazed_b200 import bamio, bcfio, datasource

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    from unfazed_b200.engine import Engine
    return Engine(0)


def _device_equals_host(engine, path, trios, regions):
    host = bcfio.read_sites(path, trios, regions)
    dev = bcfio.read_sites(path, trios, regions, engine=engine)
    assert_tables_equal(host, dev)
    assert np.array_equal(host.gq.view(np.uint32), dev.gq.view(np.uint32))
    # the fixed fields of every record of the inflated chunks, bit for bit
    bf = bcfio.BcfFile(path)
    qs = [(bf.tids[c], max(a, 0), max(b, 1)) for c, ivs in regions.items() if c in bf.tids for a, b in ivs]
    buf, offs, _ = bf.fetch_union(qs)
    want = bcfio.HostDecoder().records(buf, offs, bf.keys, len(bf.samples))
    got = engine.bcf_decoder().records(buf, offs, bf.keys, len(bf.samples))
    assert want.shape[0] > 0 and np.array_equal(want.view(np.uint8), got.view(np.uint8))
    return host, dev


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_device_equals_host_golden(engine, tmp_path, name):
    ds, _ = load_case(name)
    path = str(tmp_path / "g.bcf")
    bcfio.write_bcf(ds.sites, path)
    prefix = "chr" if ds.sites.contigs[0].startswith("chr") else ""
    _device_equals_host(engine, path, ds.sites.trios, dnm_regions(ds.dnms, prefix))


def test_device_equals_host_hand_assembled(engine, tmp_path):
    for variant in ("idx", "plain"):
        path = str(tmp_path / ("h_%s.bcf" % variant))
        write_hand_bcf(path, variant)
        _device_equals_host(engine, path, [("s0", "s1", "s2")], {"1": [(0, 1000)], "2": [(0, 1000)]})


def _assemble_large(path, head, recs, tid):
    """Like assemble, for record data over one BGZF block: the records through the repository's BGZF writer."""
    import struct
    htext = head.encode() + b"\0"
    body = b"".join(recs)
    voff = bamio.write_bgzf(path, b"BCF\x02\x02" + struct.pack("<I", len(htext)) + htext, body)
    starts = np.cumsum([0] + [len(r) for r in recs]).astype(np.int64)
    pos = np.array([struct.unpack_from("<i", r, 12)[0] for r in recs], dtype=np.int64)
    rlen = np.array([struct.unpack_from("<i", r, 16)[0] for r in recs], dtype=np.int64)
    bamio.write_csi(path + ".csi", tid + 1, np.full(len(recs), tid), pos, pos + rlen, voff(starts[:-1]), voff(starts[1:]))


def _write_random(rng, path, n_samples, n_records):
    k = KEYS["plain"]
    samples = ["s%d" % i for i in range(n_samples)]
    head = HEAD_PLAIN.split("#CHROM")[0] + "\t".join(["#CHROM", "POS", "ID", "REF", "ALT", "QUAL", "FILTER", "INFO",
                                                      "FORMAT"] + samples) + "\n"
    recs = _random_records(rng, n_samples, n_records)
    _assemble_large(path, head, recs, k["c1"])
    return samples, recs


def _random_records(rng, n_samples, n_records):
    k = KEYS["plain"]
    keys = ["GT", "GQ", "AD", "RO", "AO", "PL"]
    width = {INT8: (-120, 127, -128), INT16: (-32760, 32767, -32768), INT32: (-2 ** 31 + 8, 2 ** 31 - 1, -2 ** 31)}
    recs, pos = [], 100
    for _ in range(n_records):
        pos += int(rng.integers(1, 400))
        n_alt = int(rng.integers(1, 4))
        fmt = [f for f in keys if rng.random() < 0.8]
        rng.shuffle(fmt)
        fields = []
        for f in fmt:
            if f == "GQ" and rng.random() < 0.5:
                xs = [[FMISS if rng.random() < 0.1 else (FEOV if rng.random() < 0.05
                                                          else float(np.float32(rng.uniform(0, 99))))]
                      for _s in range(n_samples)]
                fields.append((k[f], FLOAT, 1, xs))
                continue
            typ = [INT8, INT16, INT32][int(rng.integers(0, 3))]
            lo, hi, miss = width[typ]
            cnt = {"GT": int(rng.integers(1, 4)), "GQ": 1, "RO": 1, "AD": n_alt + 1, "AO": n_alt,
                   "PL": (n_alt + 1) * (n_alt + 2) // 2 + 14}[f]          # PL: a count overflow
            vals = rng.integers(0, min(hi, 120), size=(n_samples, cnt)) if f != "GT" else \
                ((rng.integers(0, n_alt + 1, size=(n_samples, cnt)) + 1) << 1) | (rng.random((n_samples, cnt)) < 0.3)
            vals = vals.astype(np.int64)
            if f == "GT":
                vals[rng.random((n_samples, cnt)) < 0.1] = 0                  # missing allele
            else:
                if typ != INT8:
                    vals[rng.random((n_samples, cnt)) < 0.2] += 200         # values that need the width
                vals[rng.random((n_samples, cnt)) < 0.08] = miss
            ends = rng.integers(1, cnt + 1, size=n_samples)
            pad = (rng.random(n_samples) < 0.15)[:, None] & (np.arange(cnt)[None, :] >= ends[:, None])
            vals[pad] = miss + 1                                             # end of vector
            fields.append((k[f], typ, cnt, vals.tolist()))
        alleles = ["A"] + ["ACGT"[int(rng.integers(0, 4))] for _ in range(n_alt)]
        recs.append(record(k["c1"], pos, 1, alleles, n_samples, fmt=fields))
    return recs


@pytest.mark.parametrize("seed", [11, 12])
def test_device_equals_host_random_layouts_and_widths(engine, tmp_path, seed):
    rng = np.random.default_rng(seed)
    path = str(tmp_path / "r.bcf")
    samples, _ = _write_random(rng, path, 30, 400)
    trios = [tuple(samples[i: i + 3]) for i in range(0, 27, 3)]              # s27..s29 are not members
    host, _ = _device_equals_host(engine, path, trios, {"1": [(0, 10 ** 6)]})
    assert host.n_rows == 400 * len(trios)
    assert np.any(host.gt == 1) and np.any(host.ad == -1) and np.any(host.gq != np.round(host.gq))


def test_device_equals_host_3000_samples_records_over_64kb(engine, tmp_path):
    rng = np.random.default_rng(5)
    path = str(tmp_path / "big.bcf")
    samples, recs = _write_random(rng, path, 3000, 24)
    assert max(len(r) for r in recs) > 64 * 1024
    trios = [tuple(samples[i: i + 3]) for i in range(0, 3000, 3)]
    _device_equals_host(engine, path, trios, {"1": [(0, 10 ** 6)]})


def test_batch_phaser_records_from_device_decoded_sites(engine, tmp_path):
    from tests.test_bamio_cpu import CASES
    from unfazed_b200.phaser import BatchPhaser
    from unfazed_b200.synth import make_dataset
    ds = make_dataset(CASES[1])
    path = str(tmp_path / "b.bcf")
    bcfio.write_bcf(ds.sites, path)
    datasource._registry.clear()
    dev = datasource.load_sites(path, ds.dnms, ds.pedigrees, 5000, engine=engine)
    want = BatchPhaser(engine, ds.sites, ds.reads, ds.pedigrees).phase(copy.deepcopy(ds.dnms), threads=1)
    got = BatchPhaser(engine, dev, ds.reads, ds.pedigrees).phase(copy.deepcopy(ds.dnms), threads=1)
    assert set(got) == set(want) and len(want) > 0
    for k in want:
        assert got[k] == want[k], k


SV_TYPES = ("DEL", "DUP", "INV", "CNV", "DUP:TANDEM", "DEL:ME", "CPX", "CTX")


def _dnm_bcf(ds, path):
    kids = sorted({d["kid"] for d in ds.dnms})
    contigs = []
    for d in ds.dnms:
        if d["chrom"] not in contigs:
            contigs.append(d["chrom"])
    rows = []
    for d in ds.dnms:
        sv = d["vartype"] in SV_TYPES
        ref = "N" if sv else "N" * max(int(d["end"]) - int(d["start"]), 1)
        gts = [[2, 4] if k == d["kid"] else [2, 2] for k in kids]
        rows.append((contigs.index(d["chrom"]), int(d["start"]), int(d["end"]) if sv else None, ref,
                     "<%s>" % d["vartype"] if sv else "A", d["vartype"] if sv else None, gts))
    dnm_bcf(path, kids, rows, contigs)


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_cli_bed_from_bcf_and_csi_bams_without_cyvcf2_or_pysam(engine, tmp_path, name):
    from oracle.make_golden import cli_files
    from tests.test_gpu_golden import _bed_rows
    from unfazed_b200.__main__ import main
    ds, want = load_case(name)
    bed, ped, pairs = cli_files(ds, str(tmp_path))
    sites = str(tmp_path / "sites.bcf")
    bcfio.write_bcf(ds.sites, sites)
    dnm_inputs = [bed]
    if name == "sv_cnv":
        dnm_inputs.append(str(tmp_path / "dnms.bcf"))
        _dnm_bcf(ds, dnm_inputs[-1])
    datasource._registry.clear()
    saved = {m: sys.modules.get(m) for m in ("cyvcf2", "pysam")}
    sys.modules["cyvcf2"] = None                      # neither decoder may be needed
    sys.modules["pysam"] = None
    try:
        for kid, path in pairs:
            bamio.write_bam(ds.reads, ds.reads.kids.index(kid), path, index="csi")
            assert bamio.index_path(path) == path + ".csi"
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
