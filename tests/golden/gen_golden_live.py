#!/usr/bin/env python
"""Generate tests/golden/ref_live_fuzz.json.gz by running the REAL reference (pure-Python configuration) on
seeded random cases; tests/test_oracle_live_reference.py replays them against the CPU oracle.

    PYTHONHASHSEED=0 python tests/golden/gen_golden_live.py <reference checkout>

Every record holds the case (hex pattern and haystack, k or the generic limits) and, for each route the case is
eligible for, the reference's raw match stream as [count, digest] (``digest``: the same function in
tests/test_oracle_live_reference.py; raw streams of short patterns run to megabytes).  "final" is the reference's
find_near_matches list in full (ties inside a group of overlapping matches depend on set order, so the test checks
it for admissibility, not equality)."""
import gzip
import hashlib
import json
import os
import random
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SEED = 20261017

if os.environ.get("PYTHONHASHSEED") != "0":
    os.environ["PYTHONHASHSEED"] = "0"
    os.execv(sys.executable, [sys.executable] + sys.argv)

sys.path.insert(0, os.path.join(sys.argv[1], "src"))

import fuzzysearch  # noqa: E402
from fuzzysearch import generic_search, levenshtein, levenshtein_ngram, substitutions_only  # noqa: E402
from fuzzysearch.common import LevenshteinSearchParams  # noqa: E402

assert levenshtein_ngram._expand_short is levenshtein_ngram._py_expand_short, "natives present?"


def case(rng, mmax=28, nmax=220):
    alphabet = rng.choice([b"ab", b"ACGT", b"abcdefgh", bytes(range(32, 127))])
    m = rng.randint(1, mmax)
    pat = bytes(rng.choice(alphabet) for _ in range(m))
    hay = bytearray(rng.choice(alphabet) for _ in range(rng.randint(0, nmax)))
    for _ in range(rng.randint(0, 4)):
        v = bytearray(pat)
        for _ in range(rng.randint(0, 4)):
            op = rng.randrange(3)
            if op == 0 and v:
                v[rng.randrange(len(v))] = rng.choice(alphabet)
            elif op == 1:
                v.insert(rng.randrange(len(v) + 1), rng.choice(alphabet))
            elif v:
                del v[rng.randrange(len(v))]
        pos = rng.randint(0, len(hay))
        hay[pos:pos + len(v)] = v
    return pat, bytes(hay)


def t(ms):
    return [[m.start, m.end, m.dist] for m in ms]


def digest(triples):
    return [len(triples), hashlib.sha256(json.dumps(triples, separators=(",", ":")).encode()).hexdigest()[:16]]


def h(ms):
    return digest(t(ms))


def main():
    rng = random.Random(SEED)
    lev, gen = [], []
    for _ in range(1000):
        pat, hay = case(rng)
        k = rng.randint(0, 5)
        rec = {"pat": pat.hex(), "hay": hay.hex(), "k": k,
               "subs_lp": h(substitutions_only.find_near_matches_substitutions_lp(pat, hay, k))}
        if len(pat) // (k + 1) >= 1:
            rec["ngrams"] = h(levenshtein_ngram.find_near_matches_levenshtein_ngrams(pat, hay, k))
            rec["subs_ngrams"] = h(substitutions_only.find_near_matches_substitutions_ngrams(pat, hay, k))
        if len(pat) <= 12 and k <= 3:
            rec["lp"] = h(levenshtein.find_near_matches_levenshtein_linear_programming(pat, hay, k))
        if k > 0:
            rec["final"] = t(fuzzysearch.find_near_matches(pat, hay, max_l_dist=k))
        lev.append(rec)
    for _ in range(300):
        pat, hay = case(rng, 16, 80)
        subs, ins, dels = rng.randint(0, 3), rng.randint(0, 3), rng.randint(0, 3)
        l = rng.choice([None, rng.randint(0, 4)])
        params = LevenshteinSearchParams(subs, ins, dels, l)
        up = list(params.unpacked)
        rec = {"pat": pat.hex(), "hay": hay.hex(), "params": up,
               "lp": h(generic_search._find_near_matches_generic_linear_programming(pat, hay, params))}
        if len(pat) // (up[3] + 1) >= 1:
            rec["ngrams"] = h(generic_search.find_near_matches_generic_ngrams(pat, hay, params))
        gen.append(rec)
    out = {"source": "seeded cases (random.Random(%d)) through the pure-Python reference (fuzzysearch 0.8.1), "
                     "PYTHONHASHSEED=0" % SEED, "levenshtein": lev, "generic": gen}
    with gzip.GzipFile(os.path.join(HERE, "ref_live_fuzz.json.gz"), "wb", mtime=0) as f:
        f.write(json.dumps(out, separators=(",", ":")).encode())
    print("%d + %d records" % (len(lev), len(gen)))


if __name__ == "__main__":
    main()
