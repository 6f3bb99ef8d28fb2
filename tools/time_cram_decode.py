"""Cost of reading an indexed CRAM 3.0 natively (cramio) on the c2-shaped load of tools/time_bam_decode.py.

Writes one c2-shaped kid (BASELINE config[1] synthesis, --dnms DNMs, 30x 150 bp reads, NM / RG tags, one in ten reads
with an SA tag) as a BAM + BAI and as a CRAM 3.0 + CRAI (gzip blocks, 10 000 records per slice) against a random FASTA,
then reports as one JSON line:

* host_decompress_s -- CRAI query, container / slice parsing and block decompression of the load's slices
                       (CramFile.prepare, thread pool), wall time;
* cram_decoder      -- bytes up (blocks, descriptors, reference spans) and down, and CUDA-event times of the upload,
                       cram_slice_size_kernel, the scan and cram_slice_write_kernel, summed over the load;
* bam_stages_ms     -- the shared BAM stages of the same load (unfz_bam_parse, offsets, emit);
* load_reads_s      -- datasource.load_reads end to end from the CRAM: host-only decode and with the GPU decode, and from
                       the BAM of the same reads with the GPU decode.
The CRAM load is checked against the BAM load (headers, CIGARs, names, device columns).  The writer is Python, so the
default load is smaller than time_bam_decode.py's.  Needs a GPU."""
import argparse
import copy
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from unfazed_b200 import bamio, cramio, datasource  # noqa: E402
from unfazed_b200.schema import AUX_HAS_SA  # noqa: E402
from unfazed_b200.synth import SynthConfig, make_dataset  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dnms", type=int, default=200)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_cram_decode.py measures the GPU decode: no CUDA device visible")
    from unfazed_b200.engine import Engine
    out = {"workload": "c2-shaped CRAM: one kid, %d SNV DNMs, 30x 150 bp reads, search-dist 5000" % args.dnms,
           "gpu": gpu_info()}
    ds = make_dataset(SynthConfig(noise=True, seed=args.seed, dnms_per_trio=args.dnms, search_dist=5000, coverage=30.0))
    t = copy.deepcopy(ds.reads)
    rng = np.random.default_rng(args.seed)
    t.hdr["aux"] |= np.where(rng.random(t.n_reads) < 0.1, AUX_HAS_SA, 0).astype(np.uint8)
    tmp = tempfile.mkdtemp(prefix="cramdecode_")
    bam, cram, ref = (os.path.join(tmp, x) for x in ("kid.bam", "kid.cram", "ref.fa"))
    tags = bamio.encode_tag("NM", "i", 1) + bamio.encode_tag("RG", "Z", "sample1")
    bamio.write_bam(t, 0, bam, common_tags=tags)
    f = bamio.BamFile(bam)
    with open(ref, "wb") as fh:
        for name, ln in zip(f.refs, f.ref_lens):
            s = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, ln)].tobytes()
            fh.write(b">" + name.encode() + b"\n" + b"\n".join(s[i:i + 60] for i in range(0, len(s), 60)) + b"\n")
    t0 = time.perf_counter()
    cramio.write_cram(t, 0, cram, ref, common_tags=tags)
    out["write_cram_s"] = time.perf_counter() - t0
    out["bam_bytes"], out["cram_bytes"] = os.path.getsize(bam), os.path.getsize(cram)
    kid = t.kids[0]
    dnms = [dict(d, bam=cram, cram_ref=ref) for d in ds.dnms if d["kid"] == kid]
    dnms_bam = [dict(d, bam=bam) for d in ds.dnms if d["kid"] == kid]

    # CRAI + container parsing + block decompression alone (fresh file object)
    cf = cramio.CramFile(cram, ref)
    heads = {kid: cf.head_tlen(1000001)}
    regions = datasource._regions(dnms, heads, lambda k, c: c in cf.tids, 5000, 151)
    cf = cramio.CramFile(cram, ref)
    qs = [(cf.tids[c], max(a, 0), max(b, 1)) for c, ivs in regions[kid].items() for a, b in bamio._merge(ivs)]
    t0 = time.perf_counter()
    desc = cf.prepare(cf.slices_for(qs))
    out["host_decompress_s"] = time.perf_counter() - t0
    out["slices"], out["records_in_slices"], out["decompressed_bytes"] = int(desc[0].shape[0]), int(desc[6]), int(desc[1].nbytes)

    t0 = time.perf_counter()
    host = datasource.load_reads(dnms, 5000, 151, 1000000)
    out["load_reads_s"] = {"cram_host_decode": time.perf_counter() - t0}
    out["reads"], out["bases"] = host.n_reads, int(host.qual.shape[0])

    eng = Engine(0)
    datasource.load_reads(dnms[:5], 5000, 151, 1000000, engine=eng, min_gt_qual=20)     # warm-up
    datasource.load_reads(dnms_bam[:5], 5000, 151, 1000000, engine=eng, min_gt_qual=20)
    eng._cram = None
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    dev = datasource.load_reads(dnms, 5000, 151, 1000000, engine=eng, min_gt_qual=20)
    torch.cuda.synchronize()
    out["load_reads_s"]["cram_gpu_decode"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    devb = datasource.load_reads(dnms_bam, 5000, 151, 1000000, engine=eng, min_gt_qual=20)
    torch.cuda.synchronize()
    out["load_reads_s"]["bam_gpu_decode"] = time.perf_counter() - t0
    cd = eng.cram_decoder()
    out["cram_decoder"] = {"h2d_bytes": cd.h2d_bytes, "d2h_bytes": cd.d2h_bytes, "kernels_ms": dict(cd.timings_ms)}
    dec = dev.device_source
    out["bam_stages_ms"] = {k: dec.timings_ms.get(k) for k in ("parse", "concat_src", "mate_join", "emit")}
    same = (np.array_equal(dev.hdr, devb.hdr) and np.array_equal(dev.cigar, devb.cigar) and dev.names == devb.names
            and all(torch.equal(getattr(dev.device_reads, k).view(torch.uint8), getattr(devb.device_reads, k).view(torch.uint8))
                    for k in ("hdr", "cigar", "seq2", "lowq", "nmask", "start")))
    out["cram_equals_bam"] = bool(same)
    shutil.rmtree(tmp, ignore_errors=True)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
