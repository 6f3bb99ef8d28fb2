"""Cost of reading a tabix-indexed sites VCF natively (vcfio) against the cyvcf2-API packer, on c2- and c5-shaped inputs.

For each workload it writes a sorted .vcf.gz + .tbi of the synthetic site table (vcfio.write_vcf: FORMAT GT:AD:GQ, every
sample of every trio, ./. for a trio without a row in the record) and reports, in one JSON line:

* tbi_inflate_s   -- TBI parse + BGZF inflate of the union of the chunk lists of every DNM window (wall time);
* h2d             -- text bytes copied to the device and the time of that copy (CUDA events);
* kernels_ms      -- line boundaries (unfz_vcf_line_count + scan + unfz_vcf_line_write), unfz_vcf_parse and
                     unfz_vcf_samples, from CUDA events;
* d2h             -- bytes of the fixed-field records and member columns copied back, and the time of those copies;
* host_build_s    -- the host's share of a GPU load: selection, REF / ALT gathers, build_site_table;
* load_sites_s    -- datasource.load_sites end to end, host-only decode and with the GPU decode;
* pack_sites_s    -- packers.pack_sites over the oracle's cyvcf2 stand-ins on the same records;
* bound           -- which of inflate and the GPU decode takes longer in the GPU load.
The device columns are checked equal to the host decode.  Needs a GPU."""
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

from oracle import fakes  # noqa: E402
from unfazed_b200 import datasource, packers, vcfio  # noqa: E402
from unfazed_b200.synth import SynthConfig, make_dataset  # noqa: E402

FIELDS = ("blk_trio", "blk_contig", "blk_off", "pos", "flag", "ref", "alt", "gt", "gq", "rd", "ad", "rec_id")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def _equal(a, b):
    return all(np.array_equal(getattr(a, f), getattr(b, f)) for f in FIELDS) and a.extras == b.extras \
        and a.contigs == b.contigs


def workload(name, cfg, tmp, engine):
    ds = make_dataset(cfg)
    path = os.path.join(tmp, name + ".vcf.gz")
    t0 = time.perf_counter()
    vcfio.write_vcf(ds.sites, path, level=1)
    out = {"workload": name, "trios": len(ds.sites.trios), "samples": 3 * len(ds.sites.trios), "dnms": len(ds.dnms),
           "site_rows": ds.sites.n_rows, "write_vcf_s": time.perf_counter() - t0, "vcf_gz_bytes": os.path.getsize(path)}
    # TBI + inflate alone (fresh file object: nothing cached)
    vf = vcfio.VcfFile(path)
    regions = {}
    for d in ds.dnms:
        regions.setdefault(vf.prefix + d["chrom"].replace("chr", ""), []).append(
            (int(d["start"]) - cfg.search_dist - 2, int(d["end"]) + cfg.search_dist + 2))
    t0 = time.perf_counter()
    vf = vcfio.VcfFile(path)
    qs = [(vf.tids[c], max(a, 0), max(b, 1)) for c, ivs in regions.items() if c in vf.tids for a, b in vcfio._merge(ivs)]
    buf, _ = vf.fetch_union(qs)
    out["tbi_inflate_s"] = time.perf_counter() - t0
    out["text_bytes"] = int(buf.nbytes)
    del buf
    # end to end: host-only, then with the GPU (one warm-up load of each first)
    datasource._registry.clear()
    for eng, key in ((None, "host"), (engine, "gpu")):
        datasource.load_sites(path, ds.dnms, ds.pedigrees, cfg.search_dist, engine=eng)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        tab = datasource.load_sites(path, ds.dnms, ds.pedigrees, cfg.search_dist, engine=eng)
        torch.cuda.synchronize()
        out.setdefault("load_sites_s", {})[key] = time.perf_counter() - t0
        out.setdefault("rows", tab.n_rows)
        if key == "host":
            host_tab = tab
    assert _equal(host_tab, tab), "device decode differs from the host decode"
    out["device_equals_host"] = True
    # one instrumented GPU load: per-step events, bytes, the host's share
    dec = engine.vcf_decoder()
    engine.vcf_decoder = lambda: dec
    t0 = time.perf_counter()
    tab = vcfio.read_sites(path, host_tab.trios, regions, engine=engine)
    wall = time.perf_counter() - t0
    del engine.vcf_decoder
    assert _equal(host_tab, tab)
    tm = dec.timings_ms
    out["h2d"] = {"text_bytes": dec.h2d_bytes, "ms": tm.get("h2d_text", 0.0) + tm.get("h2d_select", 0.0)}
    out["kernels_ms"] = {k: tm[k] for k in ("line_bounds", "parse", "samples")}
    out["d2h"] = {"bytes": dec.d2h_bytes, "ms": tm.get("d2h_records", 0.0) + tm.get("d2h_cells", 0.0)}
    gpu_s = sum(tm.values()) / 1e3
    out["read_sites_gpu_s"] = wall
    out["host_build_s"] = wall - gpu_s - out["tbi_inflate_s"]
    out["bound"] = "inflate" if out["tbi_inflate_s"] > gpu_s else "gpu_decode"
    # the cyvcf2-API packer over the stand-ins
    fakes.register_vcf("mem://sites", ds.sites)
    t0 = time.perf_counter()
    want = packers.pack_sites(fakes.VCF("mem://sites"), host_tab.trios, regions)
    out["pack_sites_s"] = time.perf_counter() - t0
    assert _equal(want, host_tab), "vcfio differs from pack_sites"
    os.remove(path)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--c2-dnms", type=int, default=2000)
    ap.add_argument("--cohort-dnms", type=int, default=1, help="DNMs per trio of the c5-shaped cohorts")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_vcf_decode.py measures the GPU decode: no CUDA device visible")
    from unfazed_b200.engine import Engine
    engine = Engine(0)
    res = {"gpu": gpu_info(), "workloads": []}
    tmp = tempfile.mkdtemp(prefix="vcfdecode_")
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
