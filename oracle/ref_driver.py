"""TEST INFRASTRUCTURE ONLY -- runs the UNMODIFIED reference (unfazed 1.0.3) from the checkout named by
``$UNFAZED_REFERENCE``.

The reference package is imported in place (never copied) after ``oracle.fakes`` has been
installed as ``cyvcf2``/``pysam``.  It is used to generate the ``tests/golden`` fixtures
(``oracle/make_golden.py``); the tests themselves compare with those fixtures and never import it.
"""
from __future__ import annotations

import copy
import importlib
import os
import sys
from typing import Dict, List, Optional

REFERENCE_ROOT = os.environ.get("UNFAZED_REFERENCE", "")

# CLI defaults, reference __main__.py:75-223
DEFAULTS = dict(
    threads=1, build="38", no_extended=False, multiread_proc_min=1000, quiet=True,
    ab_homref=[0.0, 0.2], ab_homalt=[0.8, 1.0], ab_het=[0.2, 0.8], min_gt_qual=20, min_depth=10,
    search_dist=5000, insert_size_max_sample=1000000, stdevs=3, min_map_qual=1, readlen=151,
    split_error_margin=5, evidence_min_ratio=10,
)


def available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "unfazed"))


_mods = None


def modules():
    """Import the reference modules over the fakes; returns a namespace dict."""
    global _mods
    if _mods is not None:
        return _mods
    if not available():
        raise RuntimeError("no reference checkout at $UNFAZED_REFERENCE (%r)" % REFERENCE_ROOT)
    from . import fakes
    fakes.install()
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    names = ["utils", "site_searcher", "informative_site_finder", "read_collector",
             "snv_phaser", "sv_phaser", "unfazed"]
    _mods = {n: importlib.import_module("unfazed." + n) for n in names}
    return _mods


def register(ds) -> None:
    """Expose a synth.Dataset to the fakes under its mem:// names."""
    from . import fakes
    fakes.register_vcf(ds.vcf_name, ds.sites)
    for k, kid in enumerate(ds.reads.kids):
        fakes.register_bam(ds.bam_name(kid), ds.reads, k)


def _args(params: dict) -> dict:
    p = dict(DEFAULTS)
    p.update(params or {})
    return p


def reset_state() -> None:
    """The reference caches the insert-size estimate per kid in module globals."""
    m = modules()
    m["snv_phaser"].concordant_upper_lens.clear()
    m["sv_phaser"].concordant_upper_lens.clear()


def phase(ds, dnms: Optional[List[dict]] = None, **params) -> Dict[str, dict]:
    """Run ``phase_svs`` + ``phase_snvs`` exactly as ``unfazed()`` does (unfazed.py:585-649)."""
    m = modules()
    register(ds)
    reset_state()
    p = _args(params)
    ut = m["utils"]
    dnms = copy.deepcopy(ds.dnms if dnms is None else dnms)
    kids = list(ds.pedigrees.keys())
    snvs = [d for d in dnms if d["vartype"].upper() in ut.SNV_TYPES and d["kid"] in kids]
    svs = [d for d in dnms if d["vartype"].upper() in ut.SV_TYPES and d["kid"] in kids]
    pos = (
        kids, ds.pedigrees, ds.vcf_name, p["threads"], p["build"], p["no_extended"],
        p["multiread_proc_min"], p["quiet"], p["ab_homref"], p["ab_homalt"], p["ab_het"],
        p["min_gt_qual"], p["min_depth"], p["search_dist"], p["insert_size_max_sample"],
        p["stdevs"], p["min_map_qual"], p["readlen"], p["split_error_margin"],
    )
    phased_svs, phased_snvs = {}, {}
    if svs:
        phased_svs = m["sv_phaser"].phase_svs(svs, *pos)
    if snvs:
        phased_snvs = m["snv_phaser"].phase_snvs(snvs, *pos)
    out = phased_snvs
    out.update(phased_svs)
    return out


def find(ds, dnms: List[dict], whole_region: bool, **params):
    """``informative_site_finder.find`` with CLI defaults; returns the annotated DNM list."""
    m = modules()
    register(ds)
    p = _args(params)
    dn = copy.deepcopy(dnms)
    sd = 0 if whole_region else p["search_dist"]
    return m["informative_site_finder"].find(
        dn, ds.pedigrees, ds.vcf_name, sd, p["threads"], p["build"], p["multiread_proc_min"],
        p["quiet"], p["ab_homref"], p["ab_homalt"], p["ab_het"], p["min_gt_qual"], p["min_depth"],
        whole_region=whole_region,
    )


def summarize(records: Dict[str, dict], include_ambiguous=True, verbose=True, evidence_min_ratio=10):
    m = modules()
    out = {}
    for k, rec in records.items():
        out[k] = m["unfazed"].summarize_record(rec, include_ambiguous, verbose, evidence_min_ratio)
    return out
