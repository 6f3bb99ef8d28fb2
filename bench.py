#!/usr/bin/env python
"""Benchmark of the phasing hot path (BASELINE.json metric) -- see the contract in DESIGN.md section 7.

    python bench.py --gpus N --steps K --warmup W [--config c2]      # the CUDA path (one rank per GPU)
    python bench.py --impl reference --gpus N --steps K ...           # the reference's CPU path (oracle port)
    python bench.py ... --dump-outputs DIR                            # + the last timed step's arrays as DIR/*.npy

A step is one pass of the whole hot path (window search, site classification, read scan, read-site
allele lookup, chaining, tally, final call) over one batch of DNMs.  Workloads (BASELINE.json configs):

  c2       configs[1]: one synthetic trio, 10 000 SNV DNMs, 5 kb search-dist, 30x 150 bp reads, extended
           read-backed phasing, per-DNM ``find`` windows.  THE DEFAULT, the configuration the metric is quoted on.
  c2_many  the same trio through ``find_many`` (--multiread-proc-min 1000, the reference's default flag value)
  c3       configs[2]: 2 000 DEL/DUP/INV up to 1 Mb, allele-balance CNV phasing over interior sites + SV seeds
  c4       configs[3]: --search-dist 50000 at 60x (500 DNMs): deep chaining
  c5       configs[4]: cohort, --trios x 100 DNMs, build 38 with chrX/Y PAR autophasing.  With N ranks the ONE
           cohort is sharded by kid through unfazed_b200.shard (LPT) -> strong scaling, host gather included.

With N ranks c2..c4 give every rank its own trio of the named size (DNMs shard by kid: weak scaling, no
collective on the data path).
"""
from __future__ import annotations

import argparse
import copy
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "DNMs phased/sec"
UNIT = "DNM/s"

CONFIGS = {
    "c2": dict(label="BASELINE config[1]: synthetic trio, %(dnms)d SNV DNMs, %(sd)d bp search-dist, %(cov)gx 150bp reads, "
                     "extended read-backed phasing (per-DNM find windows)",
               synth=dict(dnms_per_trio=10000, search_dist=5000, coverage=30.0),
               run=dict(search_dist=5000, multiread_proc_min=10 ** 9)),
    "c2_many": dict(label="BASELINE config[1] through find_many (--multiread-proc-min 1000): %(dnms)d SNV DNMs, %(sd)d bp "
                          "search-dist, %(cov)gx 150bp reads",
                    synth=dict(dnms_per_trio=10000, search_dist=5000, coverage=30.0),
                    run=dict(search_dist=5000, multiread_proc_min=1000)),
    "c3": dict(label="BASELINE config[2]: synthetic SV set, %(dnms)d DEL/DUP/INV up to 1 Mb, allele-balance CNV phasing over "
                     "interior het sites + SV seed reads, %(cov)gx",
               synth=dict(dnms_per_trio=2000, search_dist=5000, coverage=30.0, sv_frac=1.0, sv_max_len=1_000_000),
               run=dict(search_dist=5000, multiread_proc_min=10 ** 9)),
    "c4": dict(label="BASELINE config[3]: long-range chaining stress, %(dnms)d SNV DNMs, --search-dist %(sd)d, %(cov)gx 150bp reads",
               synth=dict(dnms_per_trio=500, search_dist=50000, coverage=60.0),
               run=dict(search_dist=50000, multiread_proc_min=10 ** 9)),
    "c5": dict(label="BASELINE config[4]: cohort of %(trios)d trios x %(dnms)d DNMs, build 38, 5%% on chrX/Y (PAR autophasing), "
                     "%(cov)gx, sharded by kid (LPT) over the ranks",
               synth=dict(dnms_per_trio=100, search_dist=5000, coverage=30.0, sex_chrom_frac=0.05, male_frac=0.5),
               run=dict(search_dist=5000, multiread_proc_min=10 ** 9, build="38"), cohort=True),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--config", choices=sorted(CONFIGS), default="c2")
    ap.add_argument("--dnms", type=int, default=0, help="DNMs per trio (0: the config's)")
    ap.add_argument("--trios", type=int, default=200, help="c5: trios in the cohort (BASELINE names 1000; 200 keeps the "
                                                            "synthetic data generation of a default run within minutes)")
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--cpu-sample", type=int, default=0, help="DNMs in the CPU-baseline sample (0: auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--full-parity", action="store_true",
                    help="after the timed legs, phase EVERY DNM of the workload with the oracle port (all host cores) and compare "
                         "all record dicts of the timed end-to-end batch with it (N=1; adds about a minute)")
    ap.add_argument("--no-saturating", action="store_true", help="skip the 2^25-pair classifier measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed resident step returned (BatchResult arrays) as DIR/<name>.npy, "
                         "float64, so that two builds can be compared output for output on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the arrays of the CUDA path (--impl b200)")
    return args


def config_of(args):
    c = copy.deepcopy(CONFIGS[args.config])
    if args.dnms:
        c["synth"]["dnms_per_trio"] = args.dnms
    return c


def workload_config(args, world):
    c = config_of(args)
    sy = c["synth"]
    lab = c["label"] % dict(dnms=sy["dnms_per_trio"], sd=sy["search_dist"], cov=sy["coverage"], trios=args.trios)
    return {
        "workload": lab, "name": args.config, "dnms_per_trio": sy["dnms_per_trio"], "search_dist": sy["search_dist"],
        "coverage": sy["coverage"], "readlen": 150, "site_spacing_bp": 300, "noise": True,
        "trios": args.trios if c.get("cohort") else world,
        "parallelism": ("one cohort sharded by kid (LPT) x%d, host gather, no collective on the data path" % world) if c.get("cohort")
        else "shard-by-kid x%d (one trio per rank), no collective" % world,
        "l2_policy": "inputs (GBs of site/read columns) exceed the 126 MB L2; no flush needed",
    }


def make_ds(args, rank, world, n_dnms=None):
    """This rank's data.  c2..c4: one trio per rank.  c5: the trios the LPT assignment gives this rank."""
    from unfazed_b200.synth import SynthConfig, make_dataset
    c = config_of(args)
    sy = dict(c["synth"])
    if n_dnms:
        sy["dnms_per_trio"] = n_dnms
    if c.get("cohort"):
        from unfazed_b200.shard import assign_kids
        work = {"kid%d" % t: float(sy["dnms_per_trio"]) for t in range(args.trios)}
        owner = assign_kids(work, world)
        mine = tuple(t for t in range(args.trios) if owner["kid%d" % t] == rank)
        return make_dataset(SynthConfig(noise=True, seed=args.seed, trio_ids=mine, **sy))
    return make_dataset(SynthConfig(noise=True, seed=args.seed + 1000 * rank, **sy))


# ----------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML polled every 5 ms from a
    thread (the timed region of this benchmark is tens of milliseconds, too short for nvidia-smi -lms; a
    tighter poll showed up in the measurement -- NVML queries take driver locks the launches also need)."""

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.samples = []
        self.reasons = set()
        self.stop_flag = False
        self.thread = None
        self.max_mhz = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None
            return
        self.thread = threading.Thread(target=self._poll, daemon=True)
        self.thread.start()

    def _poll(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8)): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40)): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20)): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)): "sw_power_cap",
        }
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self.stop_flag:
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = int(get_reasons(self.h))
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def stop(self):
        self.stop_flag = True
        if self.thread is not None:
            self.thread.join(timeout=1)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "samples": 0, "reasons": ["nvml unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "samples": len(self.samples),
                "reasons": sorted(self.reasons)}


# ----------------------------------------------------------------------------------------------
# CPU arms (oracle port): test infrastructure timed as the reference's CPU path
# ----------------------------------------------------------------------------------------------
def port_params(args):
    from oracle import port
    run = config_of(args)["run"]
    kw = dict(threads=1, readlen=151, search_dist=run["search_dist"], multiread_proc_min=run["multiread_proc_min"])
    if "build" in run:
        kw["build"] = run["build"]
    return port.Params(**kw)


_W = {}      # state the forked CPU workers inherit


def _worker_loop(conn, idx):
    """One worker process = one reference process: ONE Phaser for the whole run, so the insert-size estimate is
    made once per kid (snv_phaser.py:14,150-154) and decoded reads stay cached across steps (warm steady state).
    The data set arrives through fork; a step is one message."""
    from oracle import port
    ds, p, shard = _W["ds"], _W["params"], _W["shards"][idx]
    ph = port.Phaser(ds.sites, ds.reads, ds.pedigrees, p)
    while True:
        if conn.recv() is None:
            return
        dn = copy.deepcopy(shard)                          # the reference annotates the DNM dicts in place
        t0 = time.perf_counter()
        recs = ph.phase(dn)
        conn.send((time.perf_counter() - t0, len(recs)))


def cpu_sample_run(ds, dnms, args):
    """One core, one warm Phaser: first pass fills the per-kid insert-size estimate and the decode cache, the
    second pass is timed (the steady state of a long reference run).  Also splits the time into site finding
    and read work for the per-stage units of BASELINE.md section 3."""
    from oracle import port
    p = port_params(args)
    ph = port.Phaser(ds.sites, ds.reads, ds.pedigrees, p)
    t0 = time.perf_counter()
    ph.phase(copy.deepcopy(dnms))
    cold = time.perf_counter() - t0
    dn = copy.deepcopy(dnms)
    t0 = time.perf_counter()
    recs = ph.phase(dn)
    warm = time.perf_counter() - t0
    snv = [d for d in copy.deepcopy(dnms) if d["vartype"].upper() in port.SNV_TYPES]
    t0 = time.perf_counter()
    if snv:
        port.find(snv, ds.pedigrees, ds.sites, p, p.search_dist, whole_region=False)
    t_find = time.perf_counter() - t0
    return recs, cold, warm, t_find


def _port_shard(idx):
    from oracle import port
    ds, p, shard = _W["ds"], _W["params"], _W["shards"][idx]
    return port.Phaser(ds.sites, ds.reads, ds.pedigrees, p).phase(copy.deepcopy(shard))


def port_all(ds, args):
    """The oracle port over EVERY DNM of the workload, sharded by kid and contiguous genomic runs over all host cores
    (forked workers: the tables are shared copy-on-write).  The checker of --full-parity, never the thing measured."""
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    by_kid = {}
    for d in ds.dnms:
        by_kid.setdefault(d["kid"], []).append(d)
    shards = []
    per = max(1, (len(ds.dnms) + 4 * cores - 1) // (4 * cores))
    many = len(ds.dnms) >= config_of(args)["run"]["multiread_proc_min"]
    for lst in by_kid.values():
        # per-DNM find windows: DNMs of a kid do not interact and a kid may be cut; in find_many mode (window
        # multiplicities count the kid's other DNMs, informative_site_finder.py:392-395) a kid stays whole and the
        # mode switch is kept by handing every shard the whole run's decision
        shards += [lst] if many else [lst[i: i + per] for i in range(0, len(lst), per)]
    prm = port_params(args)
    if many:
        prm.multiread_proc_min = 0
    _W["ds"], _W["shards"], _W["params"] = ds, shards, prm
    out = {}
    with mp.get_context("fork").Pool(cores) as pool:
        for part in pool.imap_unordered(_port_shard, range(len(shards))):
            out.update(part)
    return out


def threads_arm(ds, dnms, args):
    """The reference's own parallelism: ThreadPoolExecutor(threads) with one task per DNM (snv_phaser.py:244-298),
    threads = os.cpu_count() as north_star asks.  GIL-bound."""
    from concurrent.futures import ThreadPoolExecutor, wait
    from oracle import port
    p = port_params(args)
    ph = port.Phaser(ds.sites, ds.reads, ds.pedigrees, p)
    ph.phase(copy.deepcopy(dnms))                          # warm, as the process arm
    n_thr = os.cpu_count() or 1
    work = [[d] for d in copy.deepcopy(dnms)]
    t0 = time.perf_counter()
    with ThreadPoolExecutor(n_thr) as ex:
        wait([ex.submit(ph.phase, w) for w in work])
    dt = time.perf_counter() - t0
    return {"value": len(dnms) / dt, "unit": UNIT, "threads": n_thr, "sample": "%d DNMs, one task per DNM" % len(dnms)}


def run_reference(args):
    """The reference's CPU implementation of the path on all host cores: the oracle port (the reference itself is
    Python + cyvcf2/pysam and is not installable here), process-sharded, warm."""
    import multiprocessing as mp
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    c = config_of(args)
    full = c["synth"]["dnms_per_trio"]
    per_worker = 24 if args.config in ("c2", "c2_many", "c5") else (12 if args.config == "c3" else 4)
    n_gen = min(full * (args.trios if c.get("cohort") else 1), cores * per_worker)
    if c.get("cohort"):
        a2 = copy.copy(args)
        a2.trios = max(1, min(args.trios, (n_gen + full - 1) // full))
        ds = make_ds(a2, 0, 1)
    else:
        ds = make_ds(args, 0, 1, n_dnms=n_gen)
    shards = [ds.dnms[i::cores] for i in range(cores)]
    shards = [s for s in shards if s]
    _W["ds"], _W["shards"], _W["params"] = ds, shards, port_params(args)
    ctx = mp.get_context("fork")
    conns, procs = [], []
    for i in range(len(shards)):
        a, b = ctx.Pipe()
        pr = ctx.Process(target=_worker_loop, args=(b, i), daemon=True)
        pr.start()
        conns.append(a)
        procs.append(pr)
    times = []
    for step in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        for c_ in conns:
            c_.send(1)
        for c_ in conns:
            c_.recv()
        dt = time.perf_counter() - t0
        if step >= args.warmup:
            times.append(dt)
    for c_ in conns:
        c_.send(None)
    for pr in procs:
        pr.join(timeout=10)
    n = len(ds.dnms)
    ms = 1000.0 * float(np.mean(times))
    value = n / (ms / 1000.0)
    sample = ("%d DNMs per step (same generator and per-DNM shape as the full workload), oracle/port.py sharded over %d "
              "processes, one warm Phaser per process (insert-size estimate and decoded reads cached across steps)"
              % (n, len(shards)))
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times), "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "strong" if c.get("cohort") else "weak", "vs_baseline": None,
        "dtype": "int32/f64", "data": "synthetic", "config": workload_config(args, world), "impl": "reference",
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": len(shards), "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "scope": "DNM dicts in -> record dicts out (port.Phaser.phase), the same scope as the CUDA arm's e2e",
    }
    try:
        line["threads_arm"] = threads_arm(ds, ds.dnms[: max(2 * per_worker, 8)], args)
    except Exception as e:
        line["threads_arm"] = {"error": repr(e)}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------
# the CUDA path
# ----------------------------------------------------------------------------------------------
def _norm(rec):
    r = dict(rec)
    for k in ("dad_sites", "mom_sites", "dad_reads", "mom_reads", "cnv_dad_sites", "cnv_mom_sites"):
        if isinstance(r[k], list):
            r[k] = sorted(r[k])
    return r


def run_b200(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("cpu:gloo,cuda:nccl", device_id=torch.device("cuda", local_rank))
    from unfazed_b200.engine import Engine, make_params
    from unfazed_b200.phaser import BatchPhaser
    from unfazed_b200.plan import SNV_TYPES, SV_TYPES

    conf = config_of(args)
    runkw = dict(conf["run"])
    cohort = bool(conf.get("cohort"))
    t_gen = time.perf_counter()
    ds = make_ds(args, rank, world)
    t_gen = time.perf_counter() - t_gen
    eng = Engine(local_rank)
    dev = eng.device
    with eng.on_stream():           # CUDA events below are recorded on the stream the kernels are launched on
        _run_b200_on_stream(args, eng, ds, t_gen, conf, runkw, cohort, rank, local_rank, world)
    if world > 1:
        dist.destroy_process_group()


def _run_b200_on_stream(args, eng, ds, t_gen, conf, runkw, cohort, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    from unfazed_b200.engine import make_params
    from unfazed_b200.phaser import BatchPhaser
    from unfazed_b200.plan import SNV_TYPES, SV_TYPES
    dev = eng.device
    kids = set(ds.pedigrees)
    svs = [d for d in ds.dnms if d["vartype"].upper() in SV_TYPES and d["kid"] in kids]
    snvs = [d for d in ds.dnms if d["vartype"].upper() in SNV_TYPES and d["kid"] in kids]
    n_dnms = len(ds.dnms)

    # ---- resident leg: tables in HBM, plan made once, K steps of the kernels ------------------------------
    bp = BatchPhaser(eng, ds.sites, ds.reads, ds.pedigrees)
    params = make_params(readlen=151)
    cul = bp.cul(151, 1000000, 3)                      # insert-size estimate: once per kid per run (both arms hoist it)
    plan, layout = bp.plan_batch(snvs, svs, threads=1, build=runkw.get("build", "38"),
                                 multiread_proc_min=runkw["multiread_proc_min"], search_dist=runkw["search_dist"])

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def step_resident():
        return eng.run(bp.dsites, bp.dreads, plan, params, blk_cul=cul, download=True, keep_device=False)

    # The synthetic dataset is millions of long-lived Python objects; a generation-2 garbage collection in
    # the middle of a step costs tens of milliseconds of host time.  Collect once, then park the survivors.
    import gc
    gc.collect()
    gc.freeze()
    def steps_resident(k):
        """k steps, software-pipelined like BatchPhaser.phase_stream: the launches of the next steps are queued before
        the host waits for the download of step i (the engine rotates its arenas and pinned result blocks), so the
        host round trip of one step hides under the kernels of the next.  Every step's results reach the host."""
        from collections import deque
        pend, out = deque(), None
        for _ in range(k):
            pend.append(eng.run(bp.dsites, bp.dreads, plan, params, blk_cul=cul, download=True, keep_device=False, defer=True))
            if len(pend) > 2:                              # at most two batches queued behind the one being waited for
                out = pend.popleft().finish()
        while pend:
            out = pend.popleft().finish()
        return out

    res = step_resident()                                  # first run sizes the capacities (two host syncs)
    res = steps_resident(max(args.warmup, 3))
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    res = steps_resident(args.steps)
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(res, args.dump_outputs if rank == 0 else os.path.join(args.dump_outputs, "rank%d" % rank))
    launches_per_step = res.launches
    n_pairs, n_hits, n_reads = res.n_pairs, res.n_hits, ds.reads.n_reads
    phased = int((res.calls_strict["emitted"] == 1).sum())
    win_reads = int((res.win[1] - res.win[0]).sum() + (res.win[3] - res.win[2]).sum()) if res.win is not None else 0

    # per-kernel timings (CUDA events on the launching stream), averaged over the same K steps
    stage = {}
    for _ in range(args.steps):
        r = eng.run(bp.dsites, bp.dreads, plan, params, blk_cul=cul, time_stages=True, keep_device=False)
        for k, v in r.timings_ms.items():
            stage[k] = stage.get(k, 0.0) + v / args.steps

    # ---- end to end: the call a user makes (BatchPhaser.phase), host columns -> record dicts, every step ---
    h2d_sites = bp.dsites.nbytes
    bp.release_device()
    del bp
    torch.cuda.empty_cache()
    t_pack = time.perf_counter()
    host_reads = eng.pack_reads(ds.reads, min_gt_qual=20, pin=True)       # the columns as they cross PCIe, pinned
    t_pack = time.perf_counter() - t_pack
    host_sites = _pin_table(ds.sites)
    bpe = BatchPhaser(eng, host_sites, host_reads, ds.pedigrees, resident=False)
    bpe._cul_cache[(151, 1000000, 3)] = cul
    phase_kw = dict(threads=1, build=runkw.get("build", "38"), multiread_proc_min=runkw["multiread_proc_min"],
                    search_dist=runkw["search_dist"], readlen=151)
    if cohort and world > 1:
        phase_kw["compact"] = True        # a rank ships arrays; rank 0 builds every record dict (as the CLI's multi-GPU path)
    h2d_bytes = h2d_sites + host_reads.nbytes + plan.dnm.nbytes + plan.seg.nbytes + plan.alleles.nbytes
    d2h = {"bytes": 0}

    gather = {"ms": 0.0, "n": 0}

    def deliver(recs):
        """What ends a step: the records of the batch are on the host; in the cohort job rank 0 also holds the other
        ranks' records (what the CLI's _phase_multi_gpu does before it writes the output)."""
        if cohort and world > 1:
            t_g = time.perf_counter()
            gathered = [None] * world if rank == 0 else None
            dist.gather_object(recs, gathered, dst=0)            # CompactRecords (arrays) from every rank
            n_out = 0
            if rank == 0:
                from unfazed_b200.shard import merge_part
                merged = {}
                for g in gathered:
                    merge_part(merged, g)                        # ... become the record dicts here (native builder)
                n_out = len(merged)
            gather["ms"] += (time.perf_counter() - t_g) * 1e3
            gather["n"] += 1
            if rank == 0:
                return n_out
        return len(recs)

    # (1) one call per batch, nothing overlapped: BatchPhaser.phase(dnms)
    recs = None
    for _ in range(2):
        recs = bpe.phase(ds.dnms, **phase_kw)
        n_records = deliver(recs)
    gather["ms"], gather["n"] = 0.0, 0
    parts = {}
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        recs = bpe.phase(ds.dnms, **phase_kw)
        n_records = deliver(recs)
        for k, v in bpe.last_timing.items():
            parts[k] = parts.get(k, 0.0) + v / args.steps
    barrier()
    e2e_single_s = (time.perf_counter() - t0) / args.steps
    gather_ms = gather["ms"] / max(gather["n"], 1)
    # (2) the same K batches through BatchPhaser.phase_stream: the copies and kernels of batch k+1 are queued before the
    # host builds the records of batch k.  Every batch is uploaded, planned, run, downloaded and turned into record
    # dicts inside the timed region, exactly as in (1); only the ORDER of host and device work differs.
    for recs in bpe.phase_stream([ds.dnms] * 2, **phase_kw):
        deliver(recs)
    parts_s = {}
    barrier()
    t0 = time.perf_counter()
    for recs in bpe.phase_stream([ds.dnms] * args.steps, **phase_kw):
        n_records = deliver(recs)
        for k, v in bpe.last_timing.items():
            parts_s[k] = parts_s.get(k, 0.0) + v / args.steps
    barrier()
    e2e_s = (time.perf_counter() - t0) / args.steps
    bpe.release_device()

    ms_step = ms_total / args.steps
    t_max = torch.tensor([ms_step, e2e_s * 1000.0, e2e_single_s * 1000.0], device=dev, dtype=torch.float64)
    tot = torch.tensor([float(n_dnms), float(n_pairs), float(n_reads), float(phased), float(n_hits), float(win_reads)],
                       device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_max, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms_step, e2e_ms, e2e_single_ms = float(t_max[0]), float(t_max[1]), float(t_max[2])
    all_dnms, all_pairs, all_reads, all_phased, all_hits, all_win = (float(x) for x in tot)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
        hd = ds.reads.hdr
        n_cig, n_base = int(hd["n_cigar"].sum()), int(hd["l_seq"].sum())
        # algorithmic bytes (DESIGN.md section 3): header 32 + CIGAR 4/op + 1 bit per base in, 32 B summary out
        rs_bytes = float(32 * n_reads + 4 * n_cig + n_base / 8.0 + 32 * n_reads)
        # read-by-site allele lookup unit of SURVEY 8(d) in this format: scan bytes + 2-bit base and quality bit at
        # every hit + 4 B per hit word
        lookup_bytes = rs_bytes + float(n_hits) * (1 + 4)
        kern = {
            "classify_sites": {"ms": stage.get("classify_sites", 0.0), "bytes": 45.0 * n_pairs},
            "read_scan": {"ms": stage.get("read_scan", 0.0), "bytes": rs_bytes},
            "read_site_alleles": {"ms": stage.get("read_site_alleles", 0.0), "bytes": None},
            "chain_tally": {"ms": stage.get("chain_tally", 0.0), "bytes": None},
            "compact_sites+scan": {"ms": stage.get("compact_sites", 0.0), "bytes": None},
            "window_search+scan": {"ms": stage.get("window_search", 0.0), "bytes": None},
            "chain_size+scans": {"ms": stage.get("chain_size", 0.0), "bytes": None},
        }
        for k, v in kern.items():
            if v["bytes"] and v["ms"] > 0:
                v["gbps"] = v["bytes"] / (v["ms"] * 1e6)
                v["frac"] = v["gbps"] / peak
        sat = None
        if not args.no_saturating:
            try:
                sat = saturating_classify(eng, max(args.steps, 3))
                sat["gbps"] = sat["bytes"] / (sat["classify_ms"] * 1e6)
                sat["frac"] = sat["gbps"] / peak
                sat["pairs_per_s"] = sat["pairs"] / (sat["classify_ms"] / 1000.0)
            except Exception as e:  # keep the headline line even if the extra measurement cannot run
                sat = {"error": repr(e)}
        bw = [k for k in kern if kern[k].get("gbps")]
        dom = max(bw, key=lambda k: kern[k]["ms"]) if bw else max(kern, key=lambda k: kern[k]["ms"])
        top = max(kern, key=lambda k: kern[k]["ms"])
        domk = kern[dom]
        lookup_ms = kern["read_scan"]["ms"] + kern["read_site_alleles"]["ms"]
        traffic = None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            ent = tj.get(args.config, {}).get(dom)
            if ent and ent.get("dnms") == conf["synth"]["dnms_per_trio"]:
                traffic = ent["dram_bytes_per_launch"]
        except Exception:
            pass
        roof = {
            "kernel": dom, "bound": "hbm", "unit": "GB/s", "peak": peak, "peak_source": peak_src,
            "achieved": domk.get("gbps"), "frac": domk.get("frac"), "traffic": traffic,
            "ms_per_launch": domk["ms"], "longest_kernel": top,
            "kernels": kern, "stages_ms": {k: round(v, 4) for k, v in stage.items()},
            "classify_sites_saturating": sat,
            "read_allele_lookup": {
                "bytes": lookup_bytes, "ms": lookup_ms,
                "gbps": lookup_bytes / (lookup_ms * 1e6) if lookup_ms > 0 else None,
                "frac": lookup_bytes / (lookup_ms * 1e6) / peak if lookup_ms > 0 else None},
        }
        line = {
            "metric": METRIC, "value": all_dnms / (ms_step / 1000.0), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong" if cohort else "weak", "vs_baseline": None,
            "dtype": "int32/u8 + f64 allele balance", "data": "synthetic", "config": workload_config(args, world),
            "secondary": {
                "informative_site_pairs_classified_per_s_kernel": all_pairs / (kern["classify_sites"]["ms"] / 1000.0) if kern["classify_sites"]["ms"] > 0 else None,
                "reads_examined_per_s_kernel": all_reads / (lookup_ms / 1000.0) if lookup_ms > 0 else None,
                "pairs": all_pairs, "reads": all_reads, "hits": all_hits, "reads_in_dnm_windows": all_win,
                "dnms_with_call": all_phased, "records": n_records, "dataset_gen_s": t_gen,
            },
            "roofline": roof,
            "e2e": {"value": all_dnms / (e2e_ms / 1000.0), "unit": UNIT, "h2d_bytes_per_step": int(h2d_bytes),
                    "d2h_bytes_per_step": int(getattr(eng, "last_d2h_bytes", 0)), "ms_per_step": e2e_ms,
                    "api": "BatchPhaser.phase_stream(batches) with resident=False, one batch per step: pinned host columns -> H2D "
                           "-> window plan -> kernels -> D2H -> the record dicts phase_snvs/phase_svs return; the device work of "
                           "batch k+1 is queued before the host builds the records of batch k",
                    "breakdown_ms": dict({k: round(v, 3) for k, v in parts_s.items()}, host_gather_ms=round(gather_ms, 3)),
                    "single_call": {"value": all_dnms / (e2e_single_ms / 1000.0), "ms_per_step": e2e_single_ms,
                                    "api": "BatchPhaser.phase(dnms), one call per step, nothing overlapped",
                                    "breakdown_ms": {k: round(v, 3) for k, v in parts.items()}},
                    "one_off_pack_s": round(t_pack, 3),
                    "one_off_pack_note": "reduction of the synthetic quality bytes to the 1-bit plane + pinning; a BAM packer "
                                         "writes the plane directly"},
            "gpu_launches": int(launches_per_step * args.steps),
            "spec_fallbacks": int(getattr(eng, "spec_fallbacks", 0)),
            "clocks": clocks,
        }
        if world == 1 and not args.no_cpu_baseline:
            n_s = args.cpu_sample or {"c2": 100, "c2_many": 100, "c5": 100, "c3": 40, "c4": 8}[args.config]
            sample = ds.dnms[: min(n_s, n_dnms)]
            want, cold, warm, t_find = cpu_sample_run(ds, sample, args)
            line["cpu_baseline"] = {
                "value": len(sample) / warm, "unit": UNIT, "cores": 1, "kind": "port",
                "sample": "first %d DNMs of the same workload, oracle/port.py (pure-Python restatement of the reference), warm "
                          "second pass %.1f s (first pass incl. insert-size estimate and read decoding %.1f s), %d records"
                          % (len(sample), warm, cold, len(want)),
                "cold_value": len(sample) / cold,
                "stages": {"site_pairs_per_s_in_find": (all_pairs / all_dnms * len(sample)) / t_find if t_find > 0 else None,
                           "reads_examined_per_s": (all_win / all_dnms * len(sample)) / max(warm - t_find, 1e-9)},
            }
            # parity of the timed GPU batch against the port on the sample
            keys = {_k(d) for d in sample}
            got = {k: v for k, v in recs.items() if k in keys}
            bad = [k for k in sorted(set(want) | set(got))
                   if k not in want or k not in got or _norm(want[k]) != _norm(got[k])]
            line["parity"] = len(bad) == 0
            line["parity_detail"] = {"dnms_compared": len(sample), "records_compared": len(want), "mismatches": bad[:5]}
            if args.full_parity:
                t_fp = time.perf_counter()
                want_all = port_all(ds, args)
                bad = [k for k in sorted(set(want_all) | set(recs))
                       if k not in want_all or k not in recs or _norm(want_all[k]) != _norm(recs[k])]
                line["parity_full"] = {"ok": len(bad) == 0, "dnms_compared": n_dnms, "records_compared": len(want_all),
                                       "gpu_records": len(recs), "mismatches": bad[:5],
                                       "oracle_wall_s": round(time.perf_counter() - t_fp, 1)}
                line["parity"] = line["parity"] and len(bad) == 0
        print(json.dumps(line))


DUMP_LIMIT = 64 << 20


def dump_outputs(res, path):
    """The host arrays of a BatchResult (what Engine.run hands its caller) as float64 .npy files, exact for their
    int32/int64 values; a structured array gives one file per field (``tally.n_dad_reads``).  Should they exceed
    DUMP_LIMIT bytes in all, every array keeps the same seeded sample of its last axis."""
    arrays = {name: getattr(res, name) for name in ("seg_row_lo", "seg_pair_off", "n_het", "n_cand", "cnv_dad", "cnv_mom",
                                                     "win", "slot_off") if getattr(res, name) is not None}
    for name in ("tally", "calls_strict", "calls_ambiguous"):
        a = getattr(res, name)
        for f in a.dtype.names:
            arrays[name + "." + f] = a[f]
    total = sum(8 * a.size for a in arrays.values())
    budget = DUMP_LIMIT - 4096 * len(arrays)                 # room for the .npy headers
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64)
        if total > budget:
            n = a.shape[-1]
            keep = np.sort(np.random.default_rng(0).choice(n, max(1, n * budget // total), replace=False))
            a = a[..., keep]
        np.save(os.path.join(path, name + ".npy"), a)


def _k(d):
    return "_".join([str(d["chrom"]), str(d["start"]), str(d["end"]), d["kid"], d["vartype"]])


def saturating_classify(eng, steps, n_rows=1 << 25, rows_per_window=336):
    """Bandwidth measurement of the site classifier alone (SURVEY 8(d) "saturating variant"): the
    named configs move only 15-150 MB through it, i.e. they are launch-bound.  2^25 rows (1.5 GB of
    site columns, generated on the device) are covered once by non-overlapping DNM windows."""
    import torch
    from unfazed_b200 import _lib as L
    from unfazed_b200.engine import make_params
    from unfazed_b200.plan import Plan
    dev = eng.device
    g = torch.Generator(device=dev)
    g.manual_seed(1234)
    V = n_rows
    pos = (torch.arange(V, device=dev, dtype=torch.int32) * 3)
    flag = (torch.rand(V, device=dev, generator=g) < 0.98).to(torch.uint8)
    gt_codes = torch.tensor([0, 1, 3, 2], device=dev, dtype=torch.uint8)
    gt = gt_codes[torch.multinomial(torch.tensor([0.45, 0.35, 0.19, 0.01], device=dev), 3 * V, replacement=True, generator=g)].reshape(3, V).contiguous()
    gq = torch.where(torch.rand(3, V, device=dev, generator=g) < 0.05, torch.rand(3, V, device=dev, generator=g) * 40, torch.full((3, V), 99.0, device=dev)).to(torch.float32).contiguous()
    depth = torch.poisson(torch.full((3, V), 30.0, device=dev), generator=g).to(torch.int32)
    frac = torch.where(gt == 1, 0.5, torch.where(gt == 3, 0.99, 0.01))
    ad = torch.round(depth * frac + torch.randn(3, V, device=dev, generator=g) * 2).clamp(min=0).to(torch.int32)
    ad = torch.minimum(ad, depth).contiguous()
    rd = (depth - ad).contiguous()
    ref = torch.full((V,), 65, device=dev, dtype=torch.uint8)
    alt = torch.full((V,), 67, device=dev, dtype=torch.uint8)
    blk_off = torch.tensor([0, V], device=dev, dtype=torch.int64)

    from unfazed_b200.engine import make_site_cols, pack_site_rows

    class Raw:
        pass
    ds = Raw()
    ds.n_rows = V
    meta, rec, dep = pack_site_rows(pos, flag, gt, gq, rd, ad)
    del flag, gt, gq, rd, ad, depth, frac
    ds.keep = (pos, ref, alt, blk_off, meta, rec, dep)
    ds.cols = make_site_cols(V, 1, blk_off, pos, ref, alt, meta, rec, dep)
    n_win = V // rows_per_window
    seg = np.zeros(n_win, dtype=L.SEG_DTYPE)
    seg["sblk"] = 0
    seg["lo_pos"] = np.arange(n_win, dtype=np.int64) * rows_per_window * 3
    seg["hi_pos"] = seg["lo_pos"] + rows_per_window * 3 - 1
    seg["mult"] = 1
    seg["dnm"] = np.arange(n_win)
    seg["mode"] = L.MODE_READ
    dnm = np.zeros(n_win, dtype=L.DNM_DTYPE)
    dnm["seg_lo"] = np.arange(n_win)
    dnm["seg_hi"] = dnm["seg_lo"] + 1
    dnm["rblk"], dnm["cnv_entry"] = -1, -1
    dnm["pos"] = seg["lo_pos"] + 1
    dnm["end"] = dnm["pos"] + 1
    plan = Plan(dnm=dnm, seg=seg, alleles=np.zeros(0, np.uint8), entries=[{}] * n_win, trio=np.zeros(n_win, np.int32),
                found=np.ones(n_win, bool))
    params = make_params()
    saved = getattr(eng, "_caps", None)
    eng._caps = None
    for _ in range(3):
        eng.run(ds, None, plan, params, keep_device=False)
    ms = {}
    for _ in range(steps):
        r = eng.run(ds, None, plan, params, time_stages=True, keep_device=False)
        for k, v in r.timings_ms.items():
            ms[k] = ms.get(k, 0.0) + v / steps
    eng._caps = saved
    return {"pairs": int(r.n_pairs), "rows": V, "windows": n_win, "classify_ms": ms.get("classify_sites"),
            "compact_ms": ms.get("compact_sites"), "window_search_ms": ms.get("window_search"),
            "bytes": 45.0 * r.n_pairs}


def _pin_table(t):
    """Copy of a site table whose columns live in pinned host memory (for the end-to-end leg)."""
    import torch
    out = copy.copy(t)
    for name in ("pos", "flag", "ref", "alt", "gt", "gq", "rd", "ad"):
        a = getattr(t, name)
        setattr(out, name, torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy())
    out.__dict__.pop("_blk_index", None)
    return out


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
