"""Cost of writing the phased VCF natively from a BCF DNM list (bcfio.write_phased_vcf) on a cohort-shaped input.

The input is the cohort of time_vcf_write.py, generated from a seed: ``--samples`` samples (FORMAT GT:GQ:DP) and
``--records`` records with one or two carriers each (0/1 among 0/0), written as a BGZF .bcf; every carrier has a phasing
record (origin dad, mom or ambiguous at random).  One JSON line reports, per step:

* inflate_s          -- reading and inflating the input whole (wall time);
* walk_s             -- the record boundaries (host walk of l_shared + l_indiv);
* parse_s            -- the fixed fields, host (unfz_bcf_parse_host) and GPU (engine.BcfDecoder.records);
* edit_list_s        -- bcfio.phase_edits: candidate records, the kids' genotypes, keys, summarize_record;
* format             -- the BCF -> VCF formatting on the host (wall) and on the GPU (wall, and the CUDA-event times of
                        the edit upload, the size kernel with the scan, the write kernel and the output download);
* bgzf_s             -- BGZF compression of the output (bamio.write_bgzf);
* write_phased_vcf_s -- the whole writer, host-only and with the GPU, to a .vcf.gz;
* pcie_bytes         -- bytes up and down of the GPU path.
The device output is checked equal to the host output byte for byte.  Needs a GPU."""
import argparse
import json
import os
import shutil
import struct
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from unfazed_b200 import bamio, bcfio  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def cohort(path, n_samples, n_records, seed):
    """The DNM cohort of time_vcf_write.py as BCF 2.2 (GT int8 x 2, GQ int8, DP int8; INFO DP int32), and its phasing
    records."""
    rng = np.random.default_rng(seed)
    samples = ["S%05d" % i for i in range(n_samples)]
    pos = np.cumsum(rng.integers(50, 5000, size=n_records)) + 1000
    head = ("##fileformat=VCFv4.2\n##FILTER=<ID=PASS,Description=\"All filters passed\",IDX=0>\n"
            "##INFO=<ID=DP,Number=1,Type=Integer,Description=\"Depth\",IDX=1>\n"
            "##FORMAT=<ID=GT,Number=1,Type=String,Description=\"Genotype\",IDX=2>\n"
            "##FORMAT=<ID=GQ,Number=1,Type=Integer,Description=\"Genotype quality\",IDX=3>\n"
            "##FORMAT=<ID=DP,Number=1,Type=Integer,Description=\"Depth\",IDX=1>\n##contig=<ID=1,IDX=0>\n"
            + "\t".join(["#CHROM", "POS", "ID", "REF", "ALT", "QUAL", "FILTER", "INFO", "FORMAT"] + samples) + "\n")
    text = head.encode() + b"\0"
    records = {}
    recs = []
    for r in range(n_records):
        gq = rng.integers(10, 99, size=n_samples).astype(np.int8)
        dp = rng.integers(5, 60, size=n_samples).astype(np.int8)
        gt = np.full((n_samples, 2), 2, dtype=np.int8)
        for s in rng.choice(n_samples, size=int(rng.integers(1, 3)), replace=False).tolist():
            gt[s, 1] = 4
            o = int(rng.integers(0, 3))
            n_dad, n_mom = (3, 0) if o == 0 else (0, 3) if o == 1 else (2, 2)
            key = "1_%d_%d_%s_POINT" % (int(pos[r]) - 1, int(pos[r]), samples[s])
            records[key] = {"region": {"chrom": "1", "start": int(pos[r]) - 1, "end": int(pos[r])}, "kid": samples[s],
                            "dad": "D" + samples[s], "mom": "M" + samples[s], "vartype": "POINT",
                            "evidence_type": "READBACKED", "dad_sites": ["x"] * n_dad, "mom_sites": ["y"] * n_mom,
                            "dad_reads": ["r%d" % i for i in range(n_dad)], "mom_reads": ["q%d" % i for i in range(n_mom)],
                            "cnv_dad_sites": [], "cnv_mom_sites": []}
        shared = (struct.pack("<iiifII", 0, int(pos[r]) - 1, 1, 50.0, 2 << 16 | 1, 3 << 24 | n_samples)
                  + b"\x17.\x17A\x17C\x11\x00" + b"\x11\x01\x13" + struct.pack("<i", int(dp.astype(np.int64).sum())))
        indiv = b"\x11\x02\x21" + gt.tobytes() + b"\x11\x03\x11" + gq.tobytes() + b"\x11\x01\x11" + dp.tobytes()
        recs.append(struct.pack("<II", len(shared), len(indiv)) + shared + indiv)
    bamio.write_bgzf(path, bcfio.MAGIC + struct.pack("<I", len(text)) + text, b"".join(recs), level=1)
    return samples, records


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=2000)
    ap.add_argument("--records", type=int, default=50000)
    ap.add_argument("--seed", type=int, default=17)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_bcf_write.py measures the GPU formatter: no CUDA device visible")
    from unfazed_b200.engine import Engine
    engine = Engine(0)
    res = {"gpu": gpu_info(), "samples": args.samples, "records": args.records, "seed": args.seed}
    tmp = tempfile.mkdtemp(prefix="bcfwrite_")
    try:
        src = os.path.join(tmp, "dnms.bcf")
        t0 = time.perf_counter()
        samples, records = cohort(src, args.samples, args.records, args.seed)
        res["generate_s"] = time.perf_counter() - t0
        res["input_bgzf_bytes"] = os.path.getsize(src)
        res["phasing_records"] = len(records)
        t0 = time.perf_counter()
        text, _s, strs, contigs, buf, _o, where = bcfio._read_whole(src)
        res["inflate_s"] = time.perf_counter() - t0
        res["record_bytes"] = int(buf.nbytes)
        t0 = time.perf_counter()
        offs, _stop = bcfio.record_offsets(buf)
        res["walk_s"] = time.perf_counter() - t0
        keys = np.array([strs.get(k, -1) for k in bcfio.FORMAT_KEYS], dtype=np.int32)
        names = bcfio.dictionaries(strs, contigs)
        fkeys = np.array([strs.get(k, -1) for k in ("GT", "UOPS", "UET")], dtype=np.int32)
        outs, res["parse_s"], res["format"] = {}, {}, {}
        for key in ("host", "gpu"):
            for rep in range(2):                                     # the second of two runs is reported
                dec = engine.bcf_decoder() if key == "gpu" else bcfio.HostDecoder()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                recs = bcfio._checked_records(dec, buf, offs, keys, len(samples), where)
                torch.cuda.synchronize()
                res["parse_s"][key] = time.perf_counter() - t0
                t0 = time.perf_counter()
                edit_off, edits = bcfio.phase_edits(buf, recs, samples, strs, contigs, records, False, False, 10, dec)
                res["edit_list_s"] = time.perf_counter() - t0
                res["edits"] = int(edits.shape[0])
                if key == "gpu":
                    dec.timings_ms.clear()
                    h2d0, d2h0 = dec.h2d_bytes, dec.d2h_bytes
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                out, status = dec.format(edit_off, edits, len(samples), names, fkeys)
                torch.cuda.synchronize()
                wall = time.perf_counter() - t0
                assert not status.any()
                res["format"][key] = {"wall_s": wall}
                if key == "gpu":
                    res["format"][key]["events_ms"] = dict(dec.timings_ms)
                    res["format"][key]["h2d_bytes"] = dec.h2d_bytes - h2d0
                    res["format"][key]["d2h_bytes"] = dec.d2h_bytes - d2h0
                    res["pcie_bytes"] = {"h2d": dec.h2d_bytes, "d2h": dec.d2h_bytes}
                outs[key] = out.tobytes()
        assert outs["host"] == outs["gpu"], "device output differs from the host output"
        res["device_equals_host"] = True
        res["output_bytes"] = len(outs["host"])
        t0 = time.perf_counter()
        bamio.write_bgzf(os.path.join(tmp, "bgzf_only.vcf.gz"), b"", outs["host"])
        res["bgzf_s"] = time.perf_counter() - t0
        del outs
        res["write_phased_vcf_s"] = {}
        for key, eng in (("host", None), ("gpu", engine)):
            t0 = time.perf_counter()
            bcfio.write_phased_vcf(src, records, False, False, os.path.join(tmp, "out_%s.vcf.gz" % key), 10, eng)
            res["write_phased_vcf_s"][key] = time.perf_counter() - t0
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
