#!/usr/bin/env python
"""Generate tests/golden/ref_segments.json by running the REAL reference over seeded short reads.

Run in the build container only (the reference's source tree is absent on the GPU box):

    PYTHONHASHSEED=0 python tests/golden/gen_golden_segments.py

Each case is one primer, one set of limits and a few hundred seeded reads (DNA and ASCII, 0 to 300 bytes) with
mutated copies of the primer planted at their starts, middles and ends; the stored result of a read is what the
reference's find_near_matches returns for it.  Only inputs and outputs are stored.
"""
import json
import os
import random
import sys

REF = "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))

if os.environ.get("PYTHONHASHSEED") != "0":
    os.environ["PYTHONHASHSEED"] = "0"
    os.execv(sys.executable, [sys.executable] + sys.argv)

sys.path.insert(0, os.path.join(REF, "src"))
import fuzzysearch  # noqa: E402

LIMITS = [dict(max_l_dist=2), dict(max_l_dist=1), dict(max_l_dist=0),
          dict(max_substitutions=2, max_insertions=0, max_deletions=0),
          dict(max_substitutions=1, max_insertions=1, max_deletions=1),
          dict(max_substitutions=2, max_insertions=1, max_deletions=0, max_l_dist=2)]


def mutate(rng, s, alphabet, n):
    s = bytearray(s)
    for _ in range(n):
        op = rng.randrange(3)
        if op == 0 and s:
            s[rng.randrange(len(s))] = rng.choice(alphabet)
        elif op == 1:
            s.insert(rng.randrange(len(s) + 1), rng.choice(alphabet))
        elif s:
            del s[rng.randrange(len(s))]
    return bytes(s)


def main():
    rng = random.Random(20261017)
    cases = []
    for alphabet in (b"ACGT", bytes(range(32, 127))):
        for m in (6, 12, 20):
            for kw in LIMITS:
                primer = bytes(rng.choice(alphabet) for _ in range(m))
                reads = []
                for _ in range(60):
                    n = rng.choice([0, 1, m - 1, m, m + 2, rng.randrange(150), rng.randrange(300)])
                    r = bytearray(rng.choice(alphabet) for _ in range(n))
                    for where in (0, 1, 2):
                        v = mutate(rng, primer, alphabet, rng.randrange(4))
                        if 0 < len(v) <= n and rng.random() < 0.6:
                            pos = (0, (n - len(v)) // 2, n - len(v))[where]
                            r[pos:pos + len(v)] = v
                    reads.append(bytes(r))
                results = [[[x.start, x.end, x.dist] for x in fuzzysearch.find_near_matches(primer, r, **kw)]
                           for r in reads]
                cases.append({"pattern": primer.hex(), "kwargs": kw, "reads": [r.hex() for r in reads],
                              "results": results})
    with open(os.path.join(HERE, "ref_segments.json"), "w") as f:
        json.dump({"source": "fuzzysearch (reference, pure-Python path) find_near_matches per read",
                   "cases": cases}, f, separators=(",", ":"))
    print(len(cases), "cases,", sum(len(c["reads"]) for c in cases), "reads")


if __name__ == "__main__":
    main()
