"""Cost of writing the phased VCF natively (vcfio.write_phased_vcf) on a cohort-shaped DNM VCF.

The input is generated from a seed: ``--samples`` sample columns (FORMAT GT:GQ:DP) and ``--records`` records with one
or two carriers each (0/1 among 0/0), written as a BGZF .vcf.gz; every carrier has a phasing record (origin dad, mom or
ambiguous at random).  One JSON line reports, per step:

* inflate_s          -- reading and inflating the input whole (wall time);
* lines_s            -- line boundaries and fixed fields, host (unfz_vcf_*_host) and GPU (engine.VcfDecoder.lines);
* edit_list_s        -- vcfio.phase_edits: candidate lines, the kids' genotypes, keys, summarize_record;
* rewrite            -- the sample-column rewrite on the host (wall) and on the GPU (wall, and the CUDA-event times of
                        the edit upload, both kernels with the scan, and the output download);
* bgzf_s             -- BGZF compression of the output (bamio.write_bgzf);
* write_phased_vcf_s -- the whole writer, host-only and with the GPU, to a .vcf.gz;
* pcie_bytes         -- bytes up and down of the GPU path.
The device output is checked equal to the host output byte for byte.  Needs a GPU."""
import argparse
import gzip
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

from unfazed_b200 import bamio, vcfio  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def cohort(path, n_samples, n_records, seed):
    """A DNM VCF of n_records lines over n_samples samples, one or two carriers per line, and its phasing records."""
    rng = np.random.default_rng(seed)
    samples = ["S%05d" % i for i in range(n_samples)]
    cell = "0/0:%d:%d"
    pos = np.cumsum(rng.integers(50, 5000, size=n_records)) + 1000
    records = {}
    lines = []
    for r in range(n_records):
        gq = rng.integers(10, 99, size=n_samples)
        dp = rng.integers(5, 60, size=n_samples)
        cells = [cell % (g, d) for g, d in zip(gq.tolist(), dp.tolist())]
        for s in rng.choice(n_samples, size=int(rng.integers(1, 3)), replace=False).tolist():
            cells[s] = "0/1" + cells[s][3:]
            o = int(rng.integers(0, 3))
            n_dad, n_mom = (3, 0) if o == 0 else (0, 3) if o == 1 else (2, 2)
            key = "1_%d_%d_%s_POINT" % (int(pos[r]) - 1, int(pos[r]), samples[s])
            records[key] = {"region": {"chrom": "1", "start": int(pos[r]) - 1, "end": int(pos[r])}, "kid": samples[s],
                            "dad": "D" + samples[s], "mom": "M" + samples[s], "vartype": "POINT",
                            "evidence_type": "READBACKED", "dad_sites": ["x"] * n_dad, "mom_sites": ["y"] * n_mom,
                            "dad_reads": ["r%d" % i for i in range(n_dad)], "mom_reads": ["q%d" % i for i in range(n_mom)],
                            "cnv_dad_sites": [], "cnv_mom_sites": []}
        lines.append("1\t%d\t.\tA\tC\t50\tPASS\tDP=%d\tGT:GQ:DP\t" % (int(pos[r]), int(dp.sum())) + "\t".join(cells))
    head = "##fileformat=VCFv4.2\n##contig=<ID=1>\n" + "\t".join(
        ["#CHROM", "POS", "ID", "REF", "ALT", "QUAL", "FILTER", "INFO", "FORMAT"] + samples) + "\n"
    bamio.write_bgzf(path, head.encode(), ("\n".join(lines) + "\n").encode(), level=1)
    return samples, records


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=2000)
    ap.add_argument("--records", type=int, default=50000)
    ap.add_argument("--seed", type=int, default=17)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_vcf_write.py measures the GPU rewrite: no CUDA device visible")
    from unfazed_b200.engine import Engine
    engine = Engine(0)
    res = {"gpu": gpu_info(), "samples": args.samples, "records": args.records, "seed": args.seed}
    tmp = tempfile.mkdtemp(prefix="vcfwrite_")
    try:
        src = os.path.join(tmp, "dnms.vcf.gz")
        t0 = time.perf_counter()
        samples, records = cohort(src, args.samples, args.records, args.seed)
        res["generate_s"] = time.perf_counter() - t0
        res["input_gz_bytes"] = os.path.getsize(src)
        res["phasing_records"] = len(records)
        t0 = time.perf_counter()
        with gzip.open(src, "rb") as f:
            data = f.read()
        res["inflate_s"] = time.perf_counter() - t0
        _s, _t, _c, body, _ = vcfio._parse_header(data, src)
        buf = np.frombuffer(data, dtype=np.uint8)[body:]
        res["text_bytes"] = int(buf.nbytes)
        outs, res["lines_s"], res["rewrite"] = {}, {}, {}
        for key in ("host", "gpu"):
            for rep in range(2):                                     # the second of two runs is reported
                dec = engine.vcf_decoder() if key == "gpu" else vcfio.HostDecoder()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                recs = dec.lines(buf)
                torch.cuda.synchronize()
                res["lines_s"][key] = time.perf_counter() - t0
                t0 = time.perf_counter()
                edit_off, edits = vcfio.phase_edits(buf, recs, samples, records, False, False, 10, dec)
                res["edit_list_s"] = time.perf_counter() - t0
                res["edits"] = int(edits.shape[0])
                if key == "gpu":
                    dec.timings_ms.clear()
                    h2d0, d2h0 = dec.h2d_bytes, dec.d2h_bytes
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                out, bad = dec.rewrite(edit_off, edits, len(samples))
                torch.cuda.synchronize()
                wall = time.perf_counter() - t0
                assert not bad.any()
                res["rewrite"][key] = {"wall_s": wall}
                if key == "gpu":
                    res["rewrite"][key]["events_ms"] = dict(dec.timings_ms)
                    res["rewrite"][key]["h2d_edit_bytes"] = dec.h2d_bytes - h2d0
                    res["rewrite"][key]["d2h_bytes"] = dec.d2h_bytes - d2h0
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
            vcfio.write_phased_vcf(src, records, False, False, os.path.join(tmp, "out_%s.vcf.gz" % key), 10, eng)
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
