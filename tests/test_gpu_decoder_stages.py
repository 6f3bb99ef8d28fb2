"""GPU: what the device decoders share.  unfz_exclusive_scan_i64 writes exactly n + 1 offsets; a CRAM decode whose
record count is one below a multiple of 64 gives the host decode's records; and the decoder calls on empty input (no
lines or records, no selected rows, no members, no edits) give what the host entry points give."""
import ctypes as C

import numpy as np
import pytest
import torch

from tests.test_bcfio_cpu import assemble
from tests.test_bcfout_cpu import header, random_records
from tests.test_cramio_cpu import write_fasta
from tests.test_gpu_bam import _big_table
from tests.test_gpu_bcfout import _same as same_bcf_format
from tests.test_gpu_cram import _device_equals_host
from tests.test_gpu_vcf import _random_lines
from tests.test_gpu_vcfout import _same as same_vcf_rewrite
from unfazed_b200 import _lib as L
from unfazed_b200 import bamio, bcfio, cramio, vcfio

pytestmark = pytest.mark.gpu

CANARY = -0x5A5A5A5A5A5A5A5B


@pytest.fixture(scope="module")
def engine():
    from unfazed_b200.engine import Engine
    return Engine(0)


@pytest.mark.parametrize("n", [0, 1, 63, 2048, 2049])      # 2048 items are one scan tile, 2049 need two
def test_exclusive_scan_i64_writes_n_plus_one_offsets(engine, n):
    lens = np.random.default_rng(n).integers(0, 1 << 20, n).astype(np.int64)
    want = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(lens, out=want[1:])
    with engine.on_stream():
        din = torch.from_numpy(lens).to(engine.device) if n else torch.zeros(1, dtype=torch.int64, device=engine.device)
        out = torch.full((n + 2,), CANARY, dtype=torch.int64, device=engine.device)
        rc = engine.lib.unfz_exclusive_scan_i64(engine.ctx, din.data_ptr(), out.data_ptr(), n,
                                                engine._scan_work(n).data_ptr(), C.c_void_p(engine.stream.cuda_stream))
        got = out.cpu().numpy()
    assert rc == 0
    assert np.array_equal(got[: n + 1], want) and got[n + 1] == CANARY


@pytest.mark.parametrize("n_reads", [63, 127])
def test_cram_decode_of_one_below_a_multiple_of_64_records(engine, tmp_path, n_reads):
    t = _big_table(n_pairs=(n_reads - 3) // 2, n_long=3)
    bp = str(tmp_path / "t.bam")
    bamio.write_bam(t, 0, bp, level=1)
    f = bamio.BamFile(bp)
    ref = str(tmp_path / "t.fa")
    write_fasta(ref, f.refs, f.ref_lens)
    cp = str(tmp_path / "t.cram")
    cramio.write_cram(t, 0, cp, ref)
    assert _device_equals_host(engine, cp, ref) == n_reads


def _cells_equal(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert a[k].shape == b[k].shape and a[k].tobytes() == b[k].tobytes(), k


def test_vcf_empty_inputs(engine):
    # no lines: the newline pass, the parse and a rewrite of nothing
    empty = np.zeros(0, dtype=np.uint8)
    assert vcfio.HostDecoder().lines(empty).shape == engine.vcf_decoder().lines(empty).shape == (0,)
    out, bad = same_vcf_rewrite(engine, [], 3, {})
    assert out == [] and bad.shape == (0,)
    # lines, but no edits
    rng = np.random.default_rng(3)
    lines = _random_lines(rng, 6, 40, True)
    out, bad = same_vcf_rewrite(engine, lines, 6, {})
    assert len(out) == 40 and not bad.any()
    # no selected rows; no members; no sample columns either
    buf = np.frombuffer("".join(l + "\n" for l in lines).encode(), dtype=np.uint8)
    host, dev = vcfio.HostDecoder(), engine.vcf_decoder()
    assert host.lines(buf).tobytes() == dev.lines(buf).tobytes()
    every = np.arange(40, dtype=np.int64)
    for sel, slot_of, m in ((np.zeros(0, np.int64), np.arange(6, dtype=np.int32), 6),
                            (every, np.full(6, -1, np.int32), 0),
                            (every, np.zeros(0, np.int32), 0)):
        _cells_equal(host.samples(sel, slot_of, m, True), dev.samples(sel, slot_of, m, True))


def test_bcf_empty_inputs(engine, tmp_path):
    rng = np.random.default_rng(4)
    samples = ["s%d" % i for i in range(6)]
    recs, lines, _ = random_records(rng, samples, 40)
    p = str(tmp_path / "r.bcf")
    assemble(p, header(samples), recs, [int(l.startswith("chr2")) for l in lines], compress=False)
    # records, but no edits
    out, st = same_bcf_format(engine, p, (np.zeros(41, np.int64), np.zeros(0, L.VCF_EDIT_DTYPE)))
    assert out.tobytes().count(b"\n") == 40
    # no records: the parse and a format of nothing; then no selected rows, and no members
    _text, _s, strs, contigs, buf, offs, _where = bcfio._read_whole(p)
    keys = np.array([strs.get(k, -1) for k in bcfio.FORMAT_KEYS], np.int32)
    names = bcfio.dictionaries(strs, contigs)
    fkeys = np.array([strs.get(k, -1) for k in ("GT", "UOPS", "UET")], dtype=np.int32)
    res = []
    for dec in (bcfio.HostDecoder(), engine.bcf_decoder()):
        got = [dec.records(np.zeros(0, np.uint8), np.zeros(0, np.int64), keys, 6)]
        got += dec.format(np.zeros(1, np.int64), np.zeros(0, L.VCF_EDIT_DTYPE), 6, names, fkeys)
        n = dec.records(buf, offs, keys, 6).shape[0]
        cells = [dec.samples(np.zeros(0, np.int64), np.arange(6, dtype=np.int32)),
                 dec.samples(np.arange(n, dtype=np.int64), np.zeros(0, np.int32))]
        res.append((got, cells))
    (hgot, hcells), (dgot, dcells) = res
    assert [a.shape[0] for a in hgot] == [a.shape[0] for a in dgot] == [0, 0, 0]
    for a, b in zip(hcells, dcells):
        _cells_equal(a, b)
