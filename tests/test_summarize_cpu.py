"""CPU: `summarize_record` (the final call, `unfazed/unfazed.py:162-334`) of the drop-in module and of the
oracle port against the reference's answers (tests/golden/reference_answers.json.gz), over random evidence
records that cover every branch of the decision table (read-backed / allele-balance / contradictory /
ambiguous / autophased), for several `evidence_min_ratio` values and both flags."""
import copy
import hashlib
import json
import random

from oracle import port
from tests.golden_util import PROJECT, assert_reference_answers, canon

N_RECORDS, N_FULL, CALLS = 4000, 250, 12         # CALLS: 3 ratios x 2 include_ambiguous x 2 verbose per record


def _record(rng):
    n = lambda hi: rng.choice([0, 0, 0, 1, 2, 3, hi])
    sites = lambda k, tag: [str(rng.randint(1, 99999)) for _ in range(k)]
    reads = lambda k, tag: ["%s%d" % (tag, i) for i in range(k)]
    sex = rng.random() < 0.1
    rec = {
        "region": {"chrom": rng.choice(["1", "chrX", "22"]), "start": rng.randint(1, 10 ** 6), "end": rng.randint(1, 10 ** 6)},
        "vartype": rng.choice(["POINT", "DEL", "DUP", "INV"]),
        "kid": "kid", "dad": "dad", "mom": "mom",
        "dad_sites": sites(n(12), "d"), "mom_sites": sites(n(12), "m"),
        "dad_reads": reads(n(40), "dr"), "mom_reads": reads(n(40), "mr"),
        "cnv_dad_sites": sites(n(25), "cd"), "cnv_mom_sites": sites(n(25), "cm"),
        "evidence_type": "SEX-CHROM" if sex else rng.choice(["READBACKED", "NA", "READBACKED,NA"]),
    }
    if sex:
        rec["origin_parent"] = rng.choice(["dad", "mom"])
        rec["other_parent"] = "mom" if rec["origin_parent"] == "dad" else "dad"
    return rec


def _calls():
    rng = random.Random(2024)
    for _ in range(N_RECORDS):
        rec = _record(rng)
        for ratio in (1, 3, 10):
            for amb in (False, True):
                for verbose in (False, True):
                    yield rec, amb, verbose, ratio


def _summaries(summarize_record):
    """summarize_record on every call of the sweep; an exception is answered by its type name."""
    out = []
    for rec, amb, verbose, ratio in _calls():
        try:
            out.append(summarize_record(copy.deepcopy(rec), amb, verbose, ratio))
        except Exception as e:
            out.append({"raises": type(e).__name__})
    return out


def _stored(answers):
    """The answers to the first N_FULL records in full, and a 64-bit digest of the CALLS answers to every record."""
    answers = canon(answers)
    digest = [hashlib.sha256(json.dumps(answers[i: i + CALLS], sort_keys=True).encode()).hexdigest()[:16]
              for i in range(0, len(answers), CALLS)]
    return {"full": answers[: N_FULL * CALLS], "digest": digest}


ANSWERS = {"test_summarize_record_random": lambda ref: _stored(_summaries(ref.modules()["unfazed"].summarize_record))}


def test_summarize_record_random():
    for impl in (PROJECT.modules()["unfazed"], port):
        got = _summaries(impl.summarize_record)
        stored = _stored(got)
        for key in ("full", "digest"):
            assert_reference_answers("test_summarize_record_random", stored[key], key)
    # the sweep reached every kind of call the reference can make (AMBIGUOUS_BOTH is unreachable there: the
    # origin is only ever a single parent when READBACKED was appended with it)
    seen = {tuple(w["evidence_types"]) for w in got if w and "evidence_types" in w}
    for kind in (("READBACKED",), ("ALLELE-BALANCE",), ("READBACKED", "ALLELE-BALANCE"), ("AMBIGUOUS_READBACKED",),
                 ("AMBIGUOUS_ALLELE-BALANCE",), ("AMBIGUOUS_READBACKED", "AMBIGUOUS_ALLELE-BALANCE")):
        assert kind in seen, kind
