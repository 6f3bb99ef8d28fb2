"""Cost of reading a CSI-indexed sites BCF natively (bcfio) against the same records as a tabix-indexed .vcf.gz (vcfio),
on c2- and c5-shaped inputs and a 3000-sample cohort.

For each workload it writes a sorted .bcf + .csi and a .vcf.gz + .tbi of the synthetic site table (bcfio.write_bcf /
vcfio.write_vcf: FORMAT GT:AD:GQ, every sample of every trio) and reports, in one JSON line, for each format:

* index_inflate_s -- index parse + BGZF inflate of the union of the chunk lists of every DNM window (wall time);
* h2d             -- bytes copied to the device (record bytes and offsets, or text) and the time of those copies;
* kernels_ms      -- the decode kernels from CUDA events: unfz_bcf_parse and unfz_bcf_samples, or the text path's line
                     boundaries, unfz_vcf_parse and unfz_vcf_samples;
* d2h             -- bytes of the fixed-field records and member cells copied back, and the time of those copies;
* load_sites_s    -- datasource.load_sites end to end, host-only decode and with the GPU decode.
The device columns are checked equal to the host decode, and the BCF table equal to the text table.  Needs a GPU."""
import argparse
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

from unfazed_b200 import bcfio, datasource, vcfio  # noqa: E402
from unfazed_b200.synth import SynthConfig, make_dataset  # noqa: E402

FIELDS = ("blk_trio", "blk_contig", "blk_off", "pos", "flag", "ref", "alt", "gt", "gq", "rd", "ad", "rec_id")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def _equal(a, b):
    return all(np.array_equal(getattr(a, f), getattr(b, f)) for f in FIELDS) and a.extras == b.extras \
        and a.contigs == b.contigs and np.array_equal(a.gq.view(np.uint32), b.gq.view(np.uint32))


def _one_format(kind, path, ds, regions, search_dist, engine):
    mod, opener, dec_name = (bcfio, bcfio.BcfFile, "bcf_decoder") if kind == "bcf" else \
        (vcfio, vcfio.VcfFile, "vcf_decoder")
    out = {"file_bytes": os.path.getsize(path)}
    t0 = time.perf_counter()
    f = opener(path)
    qs = [(f.tids[c], max(a, 0), max(b, 1)) for c, ivs in regions.items() if c in f.tids for a, b in vcfio._merge(ivs)]
    got = f.fetch_union(qs)
    out["index_inflate_s"] = time.perf_counter() - t0
    out["inflated_bytes"] = int(got[0].nbytes)
    del got
    datasource._registry.clear()
    tabs = {}
    for eng, key in ((None, "host"), (engine, "gpu")):
        datasource.load_sites(path, ds.dnms, ds.pedigrees, search_dist, engine=eng)        # warm-up
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        tabs[key] = datasource.load_sites(path, ds.dnms, ds.pedigrees, search_dist, engine=eng)
        torch.cuda.synchronize()
        out.setdefault("load_sites_s", {})[key] = time.perf_counter() - t0
    assert _equal(tabs["host"], tabs["gpu"]), "%s: device decode differs from the host decode" % kind
    out["device_equals_host"] = True
    # one instrumented GPU load: per-step events and bytes
    dec = getattr(engine, dec_name)()
    setattr(engine, dec_name, lambda: dec)
    t0 = time.perf_counter()
    tab = mod.read_sites(path, tabs["host"].trios, regions, engine=engine)
    out["read_sites_gpu_s"] = time.perf_counter() - t0
    delattr(engine, dec_name)
    assert _equal(tabs["host"], tab)
    tm = dec.timings_ms
    up = ("h2d_records", "h2d_select") if kind == "bcf" else ("h2d_text", "h2d_select")
    out["h2d"] = {"bytes": dec.h2d_bytes, "ms": sum(tm.get(k, 0.0) for k in up)}
    kern = ("parse", "samples") if kind == "bcf" else ("line_bounds", "parse", "samples")
    out["kernels_ms"] = {k: tm[k] for k in kern}
    out["d2h"] = {"bytes": dec.d2h_bytes, "ms": tm.get("d2h_records", 0.0) + tm.get("d2h_cells", 0.0)}
    return out, tabs["host"]


def workload(name, cfg, tmp, engine):
    ds = make_dataset(cfg)
    bcf, vcf = os.path.join(tmp, name + ".bcf"), os.path.join(tmp, name + ".vcf.gz")
    bcfio.write_bcf(ds.sites, bcf, level=1)
    vcfio.write_vcf(ds.sites, vcf, level=1)
    out = {"workload": name, "trios": len(ds.sites.trios), "samples": 3 * len(ds.sites.trios), "dnms": len(ds.dnms),
           "site_rows": ds.sites.n_rows}
    prefix = bcfio.BcfFile(bcf).prefix
    regions = {}
    for d in ds.dnms:
        regions.setdefault(prefix + d["chrom"].replace("chr", ""), []).append(
            (int(d["start"]) - cfg.search_dist - 2, int(d["end"]) + cfg.search_dist + 2))
    out["bcf"], tb = _one_format("bcf", bcf, ds, regions, cfg.search_dist, engine)
    out["vcf_gz"], tv = _one_format("vcf", vcf, ds, regions, cfg.search_dist, engine)
    assert _equal(tb, tv), "bcfio differs from vcfio"
    out["rows"] = tb.n_rows
    os.remove(bcf)
    os.remove(vcf)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--c2-dnms", type=int, default=2000)
    ap.add_argument("--cohort-dnms", type=int, default=1, help="DNMs per trio of the c5-shaped cohorts")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_bcf_decode.py measures the GPU decode: no CUDA device visible")
    from unfazed_b200.engine import Engine
    engine = Engine(0)
    res = {"gpu": gpu_info(), "workloads": []}
    tmp = tempfile.mkdtemp(prefix="bcfdecode_")
    try:
        res["workloads"].append(workload("c2_1trio_%ddnms" % args.c2_dnms, SynthConfig(
            seed=1, dnms_per_trio=args.c2_dnms, search_dist=5000, coverage=0.1), tmp, engine))
        for trios in (200, 1000):
            res["workloads"].append(workload("c5_%dtrios_x%ddnms" % (trios, args.cohort_dnms), SynthConfig(
                seed=5, n_trios=trios, dnms_per_trio=args.cohort_dnms, search_dist=5000, coverage=0.1,
                sex_chrom_frac=0.05, chr_prefix="chr"), tmp, engine))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
