"""GPU: the BCF -> phased VCF formatter on the device (engine.BcfDecoder.format -> unfz_bcf_format_size /
unfz_bcf_format_write) gives byte for byte the output and record status of the host entry points, and the command line
writes the phased VCF of the five golden cases from a DNM .bcf with neither cyvcf2 nor pysam."""
import gzip
import sys

import numpy as np
import pytest

from tests.golden_util import CASES as GOLDEN_CASES, load_case
from tests.test_bcfio_cpu import FLOAT, assemble, th, vals
from tests.test_bcfout_cpu import GT3, ID, brec, header, hand_records, random_records
from tests.test_gpu_bcf import _dnm_bcf
from unfazed_b200 import _lib as L
from unfazed_b200 import bamio, bcfio, datasource
from unfazed_b200.unfazed import uet_code

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    from unfazed_b200.engine import Engine
    return Engine(0)


def _random_edits(rng, n_recs, n_samples):
    """About one cell in four of every record, any phase (haploid GTs included)."""
    rows = []
    for i in range(n_recs):
        for s in sorted(rng.choice(n_samples, size=max(1, n_samples // 4), replace=False).tolist()):
            rows.append((i, s, int(rng.integers(0, 3)), int(rng.integers(0, 10 ** 6)), int(rng.integers(-1, 7))))
    ed = np.zeros(len(rows), dtype=L.VCF_EDIT_DTYPE)
    for k, name in enumerate(("sample", "phase", "uops", "uet")):
        ed[name] = [r[k + 1] for r in rows]
    off = np.searchsorted(np.array([r[0] for r in rows], dtype=np.int64), np.arange(n_recs + 1)).astype(np.int64)
    return off, ed


def _same(engine, path, edits=None, seed=0):
    """Host and device output and status of every record of ``path``; returns (output, status)."""
    _text, samples, strs, contigs, buf, offs, where = bcfio._read_whole(path)
    keys = np.array([strs.get(k, -1) for k in bcfio.FORMAT_KEYS], np.int32)
    names = bcfio.dictionaries(strs, contigs)
    fkeys = np.array([strs.get(k, -1) for k in ("GT", "UOPS", "UET")], dtype=np.int32)
    res = []
    for dec in (bcfio.HostDecoder(), engine.bcf_decoder()):
        recs = bcfio._checked_records(dec, buf, offs, keys, len(samples), where)
        off, ed = edits if edits is not None else _random_edits(np.random.default_rng(seed), recs.shape[0], len(samples))
        res.append(dec.format(off, ed, len(samples), names, fkeys))
    (hout, hst), (dout, dst) = res
    assert np.array_equal(hst, dst)
    assert hout.tobytes() == dout.tobytes()
    assert dec.h2d_bytes > 0 and dec.d2h_bytes > 0
    return hout, hst


def test_device_equals_host_hand_records(engine, tmp_path):
    p = str(tmp_path / "h.bcf")
    assemble(p, header(["s0", "s1", "s2"]), hand_records(), [0, 0, 1, 1], compress=False)
    off = np.array([0, 1, 2, 2, 2], dtype=np.int64)
    ed = np.array([(0, 1, 4, 0), (0, 2, 9, 1)], dtype=L.VCF_EDIT_DTYPE)
    out, st = _same(engine, p, (off, ed))
    assert st.tolist() == [0, 0, 0, L.BCFOUT_FLOAT_HOST] and out.shape[0] > 0


@pytest.mark.parametrize("seed", [0, 1])
def test_device_equals_host_random_records(engine, tmp_path, seed):
    rng = np.random.default_rng(50 + seed)
    samples = ["s%d" % i for i in range(30)]
    recs, lines, _ = random_records(rng, samples, 300)
    p = str(tmp_path / "r.bcf")
    assemble(p, header(samples), recs, [int(l.startswith("chr2")) for l in lines], compress=False)
    out, st = _same(engine, p, seed=seed)
    # random phase edits land on haploid GTs: the same status, and no output
    assert (st & L.BCFOUT_HAPLOID).any() and out.shape[0] == 0
    # without haploid edits: every record printed, floats on both paths
    off, ed = _random_edits(rng, len(recs), 30)
    ed["phase"] = 0
    out, st = _same(engine, p, (off, ed))
    assert out.tobytes().count(b"\n") == 300
    assert (st == L.BCFOUT_FLOAT_HOST).any() and (st == 0).any()


def test_device_equals_host_3000_samples_over_64kb(engine, tmp_path):
    rng = np.random.default_rng(6)
    samples = ["s%d" % i for i in range(3000)]
    recs, lines, _ = random_records(rng, samples, 12)
    p = str(tmp_path / "w.bcf")
    assemble(p, header(samples), recs, [int(l.startswith("chr2")) for l in lines], compress=False)
    _text, _s, _st, _c, buf, offs, _w = bcfio._read_whole(p)
    assert max(np.diff(np.append(offs, buf.shape[0])).tolist()) > 64 * 1024
    off, ed = _random_edits(rng, 12, 3000)
    ed["phase"] = 0
    out, st = _same(engine, p, (off, ed))
    assert not (st & (L.BCFOUT_HAPLOID | L.BCFOUT_BAD)).any()
    assert max(len(x) for x in out.tobytes().split(b"\n")) > 64 * 1024


def test_device_equals_host_float_host_records(engine, tmp_path):
    """Records whose floats leave the exact path between records that do not: the host's text lands in its slot."""
    xs = [1e-7, 3.4e38, 2.5e6, 1e-30, 0.5, 123456.5]
    recs = []
    for i in range(40):
        v = [xs[(i + j) % len(xs)] for j in range(1 + i % 4)] if i % 3 else [0.25]
        recs.append(brec(0, 10 + i, ["A", "C"], 3, qual=v[0], info=[(ID["AF"], th(FLOAT, len(v)) + vals(FLOAT, v))],
                         fmt=GT3))
    p = str(tmp_path / "f.bcf")
    assemble(p, header(["k", "d", "m"]), recs, [0] * 40, compress=False)
    off, ed = _random_edits(np.random.default_rng(1), 40, 3)
    ed["phase"] = 0
    out, st = _same(engine, p, (off, ed))
    assert (st == L.BCFOUT_FLOAT_HOST).sum() > 10 and (st == 0).sum() > 10
    assert b"1e-07" in out.tobytes() and b"3.4e+38" in out.tobytes()


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
def test_cli_vcf_from_dnm_bcf_without_cyvcf2_or_pysam(engine, tmp_path, name):
    from oracle.make_golden import cli_files
    from unfazed_b200 import vcfio
    from unfazed_b200.__main__ import main
    ds, want = load_case(name)
    _bed, ped, pairs = cli_files(ds, str(tmp_path))
    sites = str(tmp_path / "sites.vcf.gz")
    vcfio.write_vcf(ds.sites, sites)
    dnms = str(tmp_path / "dnms.bcf")
    _dnm_bcf(ds, dnms)
    datasource._registry.clear()
    saved = {m: sys.modules.get(m) for m in ("cyvcf2", "pysam")}
    sys.modules["cyvcf2"] = None                      # neither library may be needed
    sys.modules["pysam"] = None
    try:
        kids = sorted({d["kid"] for d in ds.dnms})
        inp = {}                                      # the input cells, as _dnm_bcf writes them: 0/1 for the kid
        for d in ds.dnms:
            for k in kids:
                inp[(d["chrom"], int(d["start"]), k)] = ("0/1" if k == d["kid"] else "0/0", -1, -1)
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
