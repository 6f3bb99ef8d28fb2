"""Cost of reading an indexed BAM natively (bamio) against the pysam-API packer, on a c2-shaped input.

Writes a coordinate-sorted BAM + BAI of one c2-shaped kid (BASELINE config[1] synthesis, --dnms DNMs, 30x 150 bp reads,
every read with NM / RG tags, one in ten with an SA tag), then reports as one JSON line:

* bai_inflate_s     -- BAI parse + BGZF inflate of each DNM window's own chunk list (BamFile.fetch_records, thread pool),
                       wall time; chunks shared by windows count once per window here (inflated_bytes,
                       records_in_chunks), while a load reads their union once (h2d.record_bytes);
* h2d               -- inflated record bytes (+ offsets) copied to the device and the time of those copies (CUDA events),
                       next to the bytes the packed columns of the same reads take over PCIe (PackedReads.nbytes);
* kernels_ms        -- unfz_bam_parse and the emit step (unfz_bam_emit_cigar + unfz_read_starts + unfz_bam_emit_planes)
                       from CUDA events;
* load_reads_s      -- datasource.load_reads end to end: host-only decode, and with the GPU decode;
* pack_reads_s      -- packers.pack_reads over the oracle's pysam stand-ins on the same reads (first pass: the stand-ins
                       decode their reads lazily, as pysam would).
The device-decoded columns are checked bit for bit against the host-decoded table's upload.  Needs a GPU."""
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

from unfazed_b200 import bamio, datasource  # noqa: E402
from unfazed_b200.schema import AUX_HAS_SA  # noqa: E402
from unfazed_b200.synth import SynthConfig, make_dataset  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dnms", type=int, default=2000)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_bam_decode.py measures the GPU decode: no CUDA device visible")
    from unfazed_b200.engine import Engine, PackedReads
    out = {"workload": "c2-shaped BAM: one kid, %d SNV DNMs, 30x 150 bp reads, search-dist 5000" % args.dnms,
           "gpu": gpu_info()}
    ds = make_dataset(SynthConfig(noise=True, seed=args.seed, dnms_per_trio=args.dnms, search_dist=5000, coverage=30.0))
    t = copy.deepcopy(ds.reads)
    rng = np.random.default_rng(args.seed)
    t.hdr["aux"] |= np.where(rng.random(t.n_reads) < 0.1, AUX_HAS_SA, 0).astype(np.uint8)
    tmp = tempfile.mkdtemp(prefix="bamdecode_")
    path = os.path.join(tmp, "kid.bam")
    t0 = time.perf_counter()
    bamio.write_bam(t, 0, path, common_tags=bamio.encode_tag("NM", "i", 1) + bamio.encode_tag("RG", "Z", "sample1"))
    out["write_bam_s"] = time.perf_counter() - t0
    out["bam_bytes"] = os.path.getsize(path)
    kid = t.kids[0]
    dnms = [dict(d, bam=path) for d in ds.dnms if d["kid"] == kid]

    # BAI + inflate alone (fresh file object: nothing cached)
    f = bamio.BamFile(path)
    heads = {kid: f.head_tlen(1000001)}
    regions = datasource._regions(dnms, heads, lambda k, c: c in f.tids, 5000, 151)
    t0 = time.perf_counter()
    f = bamio.BamFile(path)
    qs = [(f.tid(c), max(a, 0), max(b, 1)) for c, ivs in regions[kid].items() for a, b in bamio._merge(ivs)]
    buf, offs = f.fetch_records(qs)
    out["bai_inflate_s"] = time.perf_counter() - t0
    out["inflated_bytes"] = int(buf.nbytes)
    out["records_in_chunks"] = int(sum(o.shape[0] for o in offs))
    del buf, offs

    # host-only decode
    t0 = time.perf_counter()
    host = datasource.load_reads(dnms, 5000, 151, 1000000)
    out["load_reads_s"] = {"host_decode": time.perf_counter() - t0}
    out["reads"] = host.n_reads
    out["bases"] = int(host.qual.shape[0])

    # GPU decode: warm up (context, modules) on a few DNMs, then the whole load
    eng = Engine(0)
    datasource.load_reads(dnms[:20], 5000, 151, 1000000, engine=eng, min_gt_qual=20)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    dev = datasource.load_reads(dnms, 5000, 151, 1000000, engine=eng, min_gt_qual=20)
    torch.cuda.synchronize()
    out["load_reads_s"]["gpu_decode"] = time.perf_counter() - t0
    dec = dev.device_source
    packed = PackedReads(host, 20)
    out["h2d"] = {"record_bytes": int(dec.h2d_bytes), "record_ms": dec.timings_ms.get("h2d_records"),
                  "record_GBps": dec.h2d_bytes / 1e6 / dec.timings_ms["h2d_records"] if dec.timings_ms.get("h2d_records") else None,
                  "headers_bytes": int(dev.device_reads.nbytes),
                  "packed_columns_bytes_same_reads": int(packed.nbytes),
                  "ratio_records_over_packed": (dec.h2d_bytes + dev.device_reads.nbytes) / max(packed.nbytes, 1)}
    out["kernels_ms"] = {"parse": dec.timings_ms.get("parse"), "emit": dec.timings_ms.get("emit"),
                         "concat_and_offsets": dec.timings_ms.get("concat_src")}
    # the emit step again, alone, a few times (planes of another threshold and back)
    reps = []
    for q in (30, 20, 30, 20, 30):
        dec.timings_ms.pop("emit", None)
        dec.device_reads(q)
        reps.append(dec.timings_ms["emit"])
    out["kernels_ms"]["emit_repeats"] = reps

    # bit for bit against the upload of the host-decoded table
    up = eng.upload_reads(host, min_gt_qual=20)
    dr = dec.device_reads(20)
    same = all(torch.equal(getattr(up, k).view(torch.uint8), getattr(dr, k).view(torch.uint8))
               for k in ("hdr", "cigar", "seq2", "lowq", "nmask", "start"))
    out["device_equals_host_upload"] = bool(same)

    # the pysam-API packer over the stand-ins, same reads
    from oracle import fakes
    fakes.install()
    dm = []
    for d in dnms:
        e = dict(d, bam="mem://kid.bam", cram_ref=None)
        dm.append(e)
    fakes.register_bam("mem://kid.bam", t, 0)
    t0 = time.perf_counter()
    ref = datasource.load_reads(dm, 5000, 151, 1000000)
    out["pack_reads_s"] = time.perf_counter() - t0
    out["pack_reads_reads"] = ref.n_reads
    out["speedup_vs_pack_reads"] = {k: out["pack_reads_s"] / v for k, v in out["load_reads_s"].items()}
    shutil.rmtree(tmp, ignore_errors=True)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
