import functools
import gzip
import importlib
import json
import os
import types

import numpy as np

from unfazed_b200.schema import SiteTable
from unfazed_b200.tableio import load_tables

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASES = ["snv_noisy", "indel_cluster_many", "sv_cnv", "sexchrom_chr", "no_extended"]

# Tests that compare the project with the reference on generated inputs keep the reference's answers in
# ANSWERS_FILE: each module below maps a test name to a function of a reference driver (``oracle.ref_driver``, or
# PROJECT for the package's own drop-in modules) that returns what that driver answers on the test's inputs.
# ``python -m oracle.make_golden`` rewrites the file from the reference.
ANSWER_MODULES = ["test_port_vs_reference", "test_readers_cpu", "test_site_searcher_cpu", "test_summarize_cpu",
                  "test_writers_cpu"]
ANSWERS_FILE = os.path.join(GOLDEN, "reference_answers.json.gz")
REFERENCE_MODULES = ["utils", "site_searcher", "informative_site_finder", "read_collector", "snv_phaser", "sv_phaser",
                     "unfazed"]
PROJECT = types.SimpleNamespace(
    modules=lambda: {n: importlib.import_module("unfazed_b200." + n) for n in REFERENCE_MODULES})


def canon(x):
    """An answer as the answers file stores it (tuples become lists, dict keys strings)."""
    return json.loads(json.dumps(x))


def by_index(x, pool):
    """``x`` with every object of ``pool`` (by identity) replaced by its index there: how answers name the reads and
    sites they return."""
    ids = {id(o): i for i, o in enumerate(pool)}

    def enc(v):
        if id(v) in ids:
            return ids[id(v)]
        if isinstance(v, dict):
            return {k: enc(w) for k, w in v.items()}
        if isinstance(v, (list, tuple)):
            return [enc(w) for w in v]
        return v
    return enc(x)


@functools.lru_cache(maxsize=None)
def _answers():
    with gzip.open(ANSWERS_FILE, "rt") as f:
        return json.load(f)


def reference_answer(test):
    return _answers()[test]


def assert_reference_answers(test, got, *keys):
    """``got`` (a list of answers) equals what the reference answered in ``test`` (under ``keys`` where the test
    stores several lists); the first differing answer is reported by its index."""
    want = reference_answer(test)
    for k in keys:
        want = want[k]
    got = canon(got)
    assert len(got) == len(want), (test, keys, len(got), len(want))
    for i, (g, w) in enumerate(zip(got, want)):
        assert g == w, (test, keys, i, g, w)


def load_case(name):
    sites, reads, meta = load_tables(os.path.join(GOLDEN, name + ".npz"))
    with open(os.path.join(GOLDEN, name + ".json")) as f:
        want = json.load(f)
    ds = types.SimpleNamespace(sites=sites, reads=reads, dnms=meta["dnms"], pedigrees=meta["pedigrees"],
                               params=meta["params"], truth=meta["truth"])
    return ds, want


def unit_vectors():
    with open(os.path.join(GOLDEN, "unit_vectors.json")) as f:
        return json.load(f)


def one_trio_table(rows):
    """SiteTable with one block; rows = list of dicts(pos, gt[3], gq[3], rd[3], ad[3])."""
    n = len(rows)
    t = SiteTable(
        trios=[("kid", "dad", "mom")], contigs=["1"], blk_trio=np.zeros(1, np.int32), blk_contig=np.zeros(1, np.int32),
        blk_off=np.array([0, n], np.int64), pos=np.array([r["pos"] for r in rows], np.int32),
        flag=np.ones(n, np.uint8), ref=np.full(n, ord("A"), np.uint8), alt=np.full(n, ord("C"), np.uint8),
        gt=np.array([r["gt"] for r in rows], np.uint8).T.copy(), gq=np.array([r["gq"] for r in rows], np.float32).T.copy(),
        rd=np.array([r["rd"] for r in rows], np.int32).T.copy(), ad=np.array([r["ad"] for r in rows], np.int32).T.copy())
    t.validate()
    return t
