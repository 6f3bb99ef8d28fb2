"""GPU: the phased VCF rewrite on the device (engine.VcfDecoder.rewrite -> unfz_vcf_rewrite_size / unfz_vcf_rewrite_write)
gives byte for byte the output and line status of the host entry points, and the command line writes the phased VCF
of the five golden cases from a DNM .vcf.gz with neither cyvcf2 nor pysam."""
import copy
import sys

import numpy as np
import pytest

from tests.golden_util import CASES as GOLDEN_CASES, load_case
from tests.test_gpu_vcf import _dnm_vcf, _random_lines
from tests.test_vcfout_cpu import parity_dataset, rewrite
from unfazed_b200 import bamio, datasource, vcfio
from unfazed_b200.unfazed import uet_code

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    from unfazed_b200.engine import Engine
    return Engine(0)


def _random_edits(rng, lines, n_samples, phase_haploid=False):
    """Random edits: about one cell in four, any phase where the GT has a separator (or also on haploid GTs)."""
    edits = {}
    for i, line in enumerate(lines):
        f = line.split("\t")
        keys = f[8].split(":")
        for s in sorted(rng.choice(n_samples, size=max(1, n_samples // 4), replace=False).tolist()):
            sub = f[9 + s].split(":") if 9 + s < len(f) else ["."]
            gt = sub[keys.index("GT")] if "GT" in keys and keys.index("GT") < len(sub) else None
            ok = gt is not None and ("/" in gt or "|" in gt)
            phase = int(rng.integers(0, 3)) if ok or phase_haploid else 0
            edits.setdefault(i, []).append((s, phase, int(rng.integers(0, 10 ** 6)), int(rng.integers(-1, 7))))
    return edits


def _same(engine, lines, n_samples, edits):
    host, hbad = rewrite(lines, n_samples, edits)
    dec = engine.vcf_decoder()
    dev, dbad = rewrite(lines, n_samples, edits, dec)
    assert np.array_equal(hbad, dbad)
    assert host == dev
    assert dec.h2d_bytes > 0 and dec.d2h_bytes > 0
    return host, hbad


def test_device_equals_host_parity_dataset(engine, tmp_path):
    path, records, _ = parity_dataset(tmp_path)
    for amb in (False, True):
        a, b = str(tmp_path / "host.vcf"), str(tmp_path / "dev.vcf")
        vcfio.write_phased_vcf(path, copy.deepcopy(records), amb, True, a, 10)
        vcfio.write_phased_vcf(path, copy.deepcopy(records), amb, True, b, 10, engine=engine)
        assert open(a, "rb").read() == open(b, "rb").read()


@pytest.mark.parametrize("seed", [0, 1])
def test_device_equals_host_random_lines(engine, seed):
    rng = np.random.default_rng(40 + seed)
    lines = _random_lines(rng, 30, 300, bool(seed))
    # some lines lose trailing sample columns, some end in CRLF
    lines = ["\t".join(l.split("\t")[: 9 + int(rng.integers(0, 30))]) if rng.random() < 0.1 else l for l in lines]
    lines = [l + "\r" if rng.random() < 0.1 else l for l in lines]
    host, bad = _same(engine, lines, 30, _random_edits(rng, lines, 30))
    assert not bad.any() and len(host) == 300
    assert any("1|0" in l for l in host) and any("0|1" in l for l in host)
    # phase edits on haploid GTs and more columns than samples: the same line status
    _, bad = _same(engine, lines, 30, _random_edits(rng, lines, 30, phase_haploid=True))
    assert bad.any()
    _, bad = _same(engine, lines, 25, _random_edits(rng, lines, 25))
    assert (bad & 1).any()


def test_device_equals_host_3000_samples_over_64kb(engine):
    rng = np.random.default_rng(6)
    lines = _random_lines(rng, 3000, 12, True)
    assert max(len(l) for l in lines) > 64 * 1024
    host, bad = _same(engine, lines, 3000, _random_edits(rng, lines, 3000))
    assert not bad.any() and all(len(l) > 64 * 1024 for l in host)


def test_device_equals_host_existing_uops_uet(engine):
    rng = np.random.default_rng(9)
    lines = []
    for line in _random_lines(rng, 20, 100, False):
        f = line.split("\t")
        keys = f[8].split(":")
        for k in ("UOPS", "UET"):
            if rng.random() < 0.7:
                at = int(rng.integers(0, len(keys) + 1))
                keys.insert(at, k)
                f[9:] = [":".join(c.split(":")[:at] + [str(int(rng.integers(-1, 9)))] + c.split(":")[at:])
                         if len(c.split(":")) >= at else c for c in f[9:]]
        f[8] = ":".join(keys)
        lines.append("\t".join(f))
    host, bad = _same(engine, lines, 20, _random_edits(rng, lines, 20))
    assert not bad.any()
    assert sum(l.split("\t")[8].count("UOPS") for l in host) == len(host)


def _cells(text):
    """{(chrom, pos0, sample): (GT, UOPS, UET)} of a phased VCF."""
    out, samples = {}, None
    for line in text.rstrip("\n").split("\n"):
        if line.startswith("#CHROM"):
            samples = line.split("\t")[9:]
        if line.startswith("#"):
            continue
        f = line.split("\t")
        keys = f[8].split(":")
        for s, cell in zip(samples, f[9:]):
            sub = dict(zip(keys, cell.split(":")))
            out[(f[0], int(f[1]) - 1, s)] = (sub["GT"], int(sub["UOPS"]), int(sub["UET"]))
    return out


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_cli_vcf_from_written_dnm_vcf_without_cyvcf2_or_pysam(engine, tmp_path, name):
    import gzip
    from oracle.make_golden import cli_files
    from unfazed_b200.__main__ import main
    ds, want = load_case(name)
    _bed, ped, pairs = cli_files(ds, str(tmp_path))
    sites = str(tmp_path / "sites.vcf.gz")
    vcfio.write_vcf(ds.sites, sites)
    dnms = str(tmp_path / "dnms.vcf.gz")
    _dnm_vcf(ds, dnms)
    datasource._registry.clear()
    saved = {m: sys.modules.get(m) for m in ("cyvcf2", "pysam")}
    sys.modules["cyvcf2"] = None                      # neither library may be needed
    sys.modules["pysam"] = None
    try:
        for kid, path in pairs:
            bamio.write_bam(ds.reads, ds.reads.kids.index(kid), path)
        p = dict(threads=1, build="38", multiread_proc_min=1000, no_extended=False)
        p.update(ds.params)
        for out_name in ("out.vcf", "out.vcf.gz"):
            for amb in (False, True):
                out = str(tmp_path / ("%s_%s" % (amb, out_name)))
                argv = ["-d", dnms, "-s", sites, "-p", ped, "--bam-pairs"] + ["%s:%s" % (k, b) for k, b in pairs] + \
                       ["-t", str(p["threads"]), "-g", p["build"], "--multiread-proc-min", str(p["multiread_proc_min"]),
                        "--quiet", "--verbose", "--outfile", out]
                if p["no_extended"]:
                    argv.append("--no-extended")
                if amb:
                    argv.append("--include-ambiguous")
                main(argv)
                raw = open(out, "rb").read()
                if out_name.endswith(".gz"):
                    assert raw.endswith(bamio.BGZF_EOF)
                    raw = gzip.decompress(raw)
                cells = _cells(raw.decode())
                inp = _cells(gzip.open(dnms, "rt").read().replace("\tGT\t", "\tGT:UOPS:UET\t").replace("0/1", "0/1:-1:-1")
                             .replace("0/0", "0/0:-1:-1"))
                rows = [l.split("\t") for l in want["cli"]["ambiguous" if amb else "strict"].strip().split("\n")
                        if l and not l.startswith("#")]
                assert rows
                phased = {}
                for r in rows:
                    chrom, start, kid, origin = r[0], int(r[1]), r[4], r[5]
                    ped_k = ds.pedigrees[kid]
                    gt = "1|0" if origin == ped_k["dad"] else "0|1" if origin == ped_k["mom"] else "0/1"
                    phased[(chrom, start, kid)] = (gt, int(r[7]), uet_code(r[8].split(",")))
                for k, v in cells.items():
                    assert v == phased.get(k, inp[k]), (name, out_name, amb, k)
                assert sum(v != inp[k] for k, v in cells.items()) == len(phased)
    finally:
        for m, v in saved.items():
            if v is None:
                sys.modules.pop(m, None)
            else:
                sys.modules[m] = v
        datasource._registry.clear()
