"""CPU: the oracle port against what the UNMODIFIED reference, run over the in-memory cyvcf2/pysam fakes,
phased on seeds that are not in the golden set (answers stored in tests/golden/reference_answers.json.gz)."""
import copy

import pytest

from oracle import port
from tests.golden_util import canon, reference_answer
from tests.util import norm_record, port_params
from unfazed_b200.synth import SynthConfig, make_dataset

# the read-name columns of a summary are a joined Python set in the reference (Q23): not compared
_SET_ORDERED = ("origin_parent_reads", "other_parent_reads")


def _without_read_names(summary):
    return {k: v for k, v in summary.items() if k not in _SET_ORDERED}


CASES = [
    (SynthConfig(dnms_per_trio=12, seed=201, coverage=24.0), {}),
    (SynthConfig(dnms_per_trio=12, seed=202, coverage=24.0, cluster_frac=0.4, indel_frac=0.3), {"multiread_proc_min": 1}),
    (SynthConfig(dnms_per_trio=10, seed=203, coverage=24.0, sv_frac=0.6, sv_max_len=30000), {}),
    (SynthConfig(dnms_per_trio=10, seed=204, coverage=24.0, n_trios=2, sex_chrom_frac=0.3, male_frac=1.0, chr_prefix="chr"),
     {"multiread_proc_min": 1, "threads": 2}),
    (SynthConfig(dnms_per_trio=10, seed=205, coverage=24.0), {"min_gt_qual": 30, "min_depth": 20, "ab_het": [0.3, 0.7], "readlen": 150}),
    # a wider sweep of the knobs that change control flow in the reference
    (SynthConfig(dnms_per_trio=10, seed=206, coverage=20.0), {"no_extended": True}),
    (SynthConfig(dnms_per_trio=10, seed=207, coverage=20.0, sv_frac=0.7, sv_max_len=200000), {"multiread_proc_min": 1, "threads": 2}),
    (SynthConfig(dnms_per_trio=10, seed=208, coverage=20.0, sv_frac=0.5, sv_max_len=5000, indel_frac=0.3), {"no_extended": True}),
    (SynthConfig(dnms_per_trio=8, seed=209, coverage=30.0, search_dist=1500), {"search_dist": 1500}),
    (SynthConfig(dnms_per_trio=6, seed=210, coverage=16.0, search_dist=12000, site_spacing=150), {"search_dist": 12000}),
    (SynthConfig(dnms_per_trio=10, seed=211, coverage=20.0, noise=False), {"evidence_min_ratio": 3}),
    (SynthConfig(dnms_per_trio=8, seed=212, coverage=20.0, n_trios=3, cluster_frac=0.6), {"multiread_proc_min": 1}),
    (SynthConfig(dnms_per_trio=10, seed=213, coverage=20.0, sex_chrom_frac=0.5, male_frac=0.5), {"build": "37"}),
    (SynthConfig(dnms_per_trio=10, seed=214, coverage=20.0, indel_frac=0.8), {"min_map_qual": 30, "split_error_margin": 10}),
    (SynthConfig(dnms_per_trio=8, seed=215, coverage=20.0, sv_frac=0.9, sv_max_len=1000000), {}),
]


def _phased(ref):
    """Per case: the records ``ref.phase`` returns (list fields sorted) and their verbose summaries."""
    out = {}
    for cfg, params in CASES:
        ds = make_dataset(cfg)
        recs = ref.phase(ds, **params)
        summ = ref.summarize(copy.deepcopy(recs))
        out[str(cfg.seed)] = {"records": {k: norm_record(r) for k, r in recs.items()},
                              "summary": {k: _without_read_names(v) for k, v in summ.items()}}
    return out


ANSWERS = {"test_port_equals_reference": _phased}


@pytest.mark.parametrize("cfg,params", CASES, ids=[str(c[0].seed) for c in CASES])
def test_port_equals_reference(cfg, params):
    want = reference_answer("test_port_equals_reference")[str(cfg.seed)]
    ds = make_dataset(cfg)
    ph = port.Phaser(ds.sites, ds.reads, ds.pedigrees, port_params(**params))
    got = ph.phase(copy.deepcopy(ds.dnms))
    assert set(got) == set(want["records"])
    for k, rec in want["records"].items():
        assert canon(norm_record(got[k])) == rec, k
        summary = port.summarize_record(copy.deepcopy(got[k]), True, True, 10)
        assert canon(_without_read_names(summary)) == want["summary"][k], k
