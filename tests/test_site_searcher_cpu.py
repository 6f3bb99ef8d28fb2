"""CPU: the per-variant interface mirror `unfazed_b200.site_searcher` against the reference's
`unfazed/site_searcher.py` on random inputs (the order pivot / right run / left run of `binary_search`, Q16,
and the parent-consistency filter of `match_informative_sites`), `informative_site_finder.autophaseable`
against the reference's PAR tables, and the per-variant callables of the phaser modules.  The reference's
answers are stored in tests/golden/reference_answers.json.gz; reads and sites are named by their index."""
import copy
import random
import types

from tests.golden_util import PROJECT, assert_reference_answers, by_index


def _sites(rng, n):
    pos = sorted(rng.sample(range(0, 3000), n)) if n else []
    if n > 3 and rng.random() < 0.5:                       # duplicate positions (overlapping windows, Q9)
        pos = sorted(pos + [pos[n // 2], pos[n // 3]])
    return [{"pos": p, "ref_parent": rng.choice(["dad", "mom"]), "alt_parent": rng.choice(["dad", "mom"]),
             "ref_allele": "A", "alt_allele": "C"} for p in pos]


def _binary_search(ref):
    binary_search = ref.modules()["site_searcher"].binary_search
    rng = random.Random(7)
    out = []
    for _ in range(3000):
        sites = _sites(rng, rng.randint(0, 40))
        a = rng.randint(-50, 3050)
        b = a + rng.choice([0, 1, 2, 30, 151, 400, 2000])
        out.append(by_index(binary_search(a, b, sites), sites))
    return out


def _match_informative_sites(ref):
    match_informative_sites = ref.modules()["site_searcher"].match_informative_sites
    rng = random.Random(11)
    out = []
    for _ in range(300):
        sites = _sites(rng, rng.randint(1, 30))
        reads = {}
        for hap in ("ref", "alt"):
            lst = []
            for _r in range(rng.randint(0, 12)):
                st = rng.randint(0, 2900)
                lst.append(types.SimpleNamespace(reference_start=st, reference_end=st + rng.choice([1, 50, 151, 600])))
            reads[hap] = lst
        out.append(by_index(match_informative_sites(reads, sites), sites + reads["ref"] + reads["alt"]))
    return out


def _autophaseable(ref):
    autophaseable = ref.modules()["informative_site_finder"].autophaseable
    peds = {"boy": {"kid": "boy", "dad": "d", "mom": "m", "sex": "1"}, "girl": {"kid": "girl", "dad": "d", "mom": "m", "sex": "2"}}
    rng = random.Random(5)
    edges = [10000, 10001, 60001, 2699520, 2699521, 2781479, 2781480, 154931044, 155260560, 155701383, 156030895,
             57227415, 59034050, 59363566, 56887903]
    out = []
    for build in ("37", "38", 37, 38, "19"):
        for chrom in ("X", "Y", "chrX", "chrY", "x", "7", "chr7"):
            for kid in ("boy", "girl"):
                for start in edges + [rng.randint(1, 160000000) for _ in range(6)]:
                    dn = {"chrom": chrom, "start": start, "end": start + 1, "kid": kid, "vartype": "POINT"}
                    try:
                        out.append(bool(autophaseable(dict(dn), peds, build)))
                    except Exception as e:                # e.g. an unknown build in the reference's tables
                        out.append({"raises": type(e).__name__})
    return out


class _Read:
    def __init__(self, start, seq, gaps):
        self.reference_start, self.query_sequence, self._gaps = start, seq, gaps

    def get_reference_positions(self, full_length=False):
        out, p = [], self.reference_start
        for i in range(len(self.query_sequence)):
            if i in self._gaps:
                out.append(None)
            else:
                out.append(p)
                p += 1
        return out if full_length else [x for x in out if x is not None]


def _phase_by_reads_and_snvs(ref):
    """snv_phaser.phase_by_reads, sv_phaser.phase_by_reads and sv_phaser.phase_by_snvs on random matches (truth
    table snv_phaser.py:52-69, CNV votes sv_phaser.py:71-85)."""
    mods = ref.modules()
    rng = random.Random(13)
    out = []
    for _ in range(200):
        sites = _sites(rng, rng.randint(1, 12))
        for s in sites:
            s["ref_allele"], s["alt_allele"] = rng.sample("ACGT", 2)
            s["ref_parent"], s["alt_parent"] = rng.sample(["dad", "mom"], 2)      # a trio: the two parents, either way round
            s["kid_allele"] = rng.choice(["ref_parent", "alt_parent"])
        matches, reads = {}, []
        for hap in rng.choice([("ref", "alt"), ("alt", "ref")]):
            lst = []
            for _r in range(rng.randint(0, 6)):
                st = rng.randint(0, 2900)
                rd = _Read(st, "".join(rng.choice("ACGTN") for _ in range(120)), set(rng.sample(range(120), rng.randint(0, 6))))
                reads.append(rd)
                lst.append({"read": rd, "matches": rng.sample(sites, rng.randint(0, len(sites)))})
            matches[hap] = lst
        out.append(by_index([mods["snv_phaser"].phase_by_reads(matches), mods["sv_phaser"].phase_by_reads(matches),
                             mods["sv_phaser"].phase_by_snvs(sites)], sites + reads))
    return out


def _autophase_and_get_refalt(ref):
    """``autophase`` of both phaser modules (snv_phaser.py:302-352 returns True and writes the SEX-CHROM record,
    sv_phaser.py:304-354 writes it and returns None) with the record it writes, fields in order, and ``get_refalt``
    (snv_phaser.py:73-84) over the in-memory cyvcf2 stand-in."""
    mods = ref.modules()
    from oracle import fakes
    from unfazed_b200.synth import SynthConfig, make_dataset
    peds = {"boy": {"kid": "boy", "dad": "d", "mom": "m", "sex": "1"}, "girl": {"kid": "girl", "dad": "d", "mom": "m", "sex": "2"}}
    rng = random.Random(17)
    starts = [10000, 10001, 60001, 2699520, 2699521, 2781479, 154931044, 155260560, 156030895, 59363566] + \
             [rng.randint(1, 160000000) for _ in range(10)]
    out = {"autophase": [], "get_refalt": []}
    for build in ("37", "38", "19", 38):
        for chrom in ("X", "chrY", "y", "7"):
            for kid in ("boy", "girl"):
                for start in starts:
                    dn = {"chrom": chrom, "start": start, "end": start + 1, "kid": kid, "vartype": rng.choice(["POINT", "DEL"])}
                    for name in ("snv_phaser", "sv_phaser"):
                        rec = {}
                        ret = mods[name].autophase(copy.deepcopy(dn), peds, rec, "d", "m", build)
                        out["autophase"].append([ret, [[k, list(v.items())] for k, v in rec.items()]])
    ds = make_dataset(SynthConfig(dnms_per_trio=30, n_trios=2, seed=23, coverage=1.0, chr_prefix="chr"))
    fakes.install()
    fakes.register_vcf("mem://refalt.vcf", ds.sites)
    import cyvcf2
    s = ds.sites
    probes = [(s.contigs[int(s.blk_contig[b])], int(s.pos[int(s.blk_off[b]) + k])) for b in range(s.n_blocks)
              for k in range(0, int(s.blk_off[b + 1] - s.blk_off[b]), 97)][:60]
    for contig, pos in probes:
        for chrom in (contig, contig.replace("chr", "")):
            for p in (pos, pos + 1, pos - 1, str(pos + 1)):
                out["get_refalt"].append(mods["snv_phaser"].get_refalt(chrom, p, cyvcf2.VCF("mem://refalt.vcf"), 0))
    return out


ANSWERS = {
    "test_binary_search_random": _binary_search,
    "test_match_informative_sites_random": _match_informative_sites,
    "test_autophaseable_matches_reference": _autophaseable,
    "test_phase_by_reads_and_phase_by_snvs_random": _phase_by_reads_and_snvs,
    "test_autophase_and_get_refalt_match_the_reference": _autophase_and_get_refalt,
}


def test_binary_search_random():
    assert_reference_answers("test_binary_search_random", _binary_search(PROJECT))


def test_match_informative_sites_random():
    assert_reference_answers("test_match_informative_sites_random", _match_informative_sites(PROJECT))


def test_autophaseable_matches_reference():
    assert_reference_answers("test_autophaseable_matches_reference", _autophaseable(PROJECT))


def test_phase_by_reads_and_phase_by_snvs_random():
    assert_reference_answers("test_phase_by_reads_and_phase_by_snvs_random", _phase_by_reads_and_snvs(PROJECT))


def test_autophase_and_get_refalt_match_the_reference():
    got = _autophase_and_get_refalt(PROJECT)
    for key in ("autophase", "get_refalt"):
        assert_reference_answers("test_autophase_and_get_refalt_match_the_reference", got[key], key)
    # eight lookups per probe; the sixth is the contig without its prefix at pos + 1
    assert any(ref is not None for ref, _alts in got["get_refalt"][5::8])
