"""Fuzz of the CPU oracle against the REAL reference: seeded random cases whose reference answers are stored in
tests/golden/ref_live_fuzz.json.gz (tests/golden/gen_golden_live.py).  Complements ref_fuzz.json with other
case shapes (patterns up to 28 symbols, haystacks up to 220 bytes, every route a case is eligible for).  Raw
streams are stored as [count, digest], final lists in full."""
import gzip
import hashlib
import json
import os

import pytest

import oracle
from parity import assert_final_parity, tup

FIXTURE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_live_fuzz.json.gz")


def digest(triples):
    triples = [list(x) for x in triples]
    return [len(triples), hashlib.sha256(json.dumps(triples, separators=(",", ":")).encode()).hexdigest()[:16]]


@pytest.fixture(scope="module")
def ref():
    with gzip.open(FIXTURE) as f:
        return json.loads(f.read())


def test_live_fuzz_against_reference(ref):
    assert len(ref["levenshtein"]) == 1000 and len(ref["generic"]) == 300
    for rec in ref["levenshtein"]:
        pat, hay, k = bytes.fromhex(rec["pat"]), bytes.fromhex(rec["hay"]), rec["k"]
        ctx = (pat, hay, k)
        assert ("ngrams" in rec) == (len(pat) // (k + 1) >= 1), ctx
        if "ngrams" in rec:
            assert digest(tup(oracle.levenshtein_ngrams_raw(pat, hay, k))) == rec["ngrams"], ctx
            assert digest(tup(oracle.subs_ngrams(pat, hay, k))) == rec["subs_ngrams"], ctx
        if "lp" in rec:
            assert digest(tup(oracle.levenshtein_lp_raw(pat, hay, k))) == rec["lp"], ctx
        assert digest(tup(oracle.subs_lp(pat, hay, k))) == rec["subs_lp"], ctx
        if k > 0:
            final, raw = oracle.find_near_matches(pat, hay, max_l_dist=k, return_raw=True)
            assert_final_parity(final, [tuple(x) for x in rec["final"]], raw, repr(ctx))
    for rec in ref["generic"]:
        pat, hay, up = bytes.fromhex(rec["pat"]), bytes.fromhex(rec["hay"]), rec["params"]
        assert digest(tup(oracle.generic_lp_raw(pat, hay, *up))) == rec["lp"], (pat, hay, up)
        if len(pat) // (up[3] + 1) >= 1:
            assert digest(tup(oracle.generic_ngrams_raw(pat, hay, *up))) == rec["ngrams"], (pat, hay, up)
