"""One pattern over many sequences (fzb_search_segments / find_near_matches_in_sequences) on the device.

Every segment must come out exactly as if it had been searched alone: per-segment FINAL lists tie-aware equal to the
oracle's, per-segment RAW lists equal to the oracle's raw stream as multisets, for every route, at the segment lengths
where the clipping rules bite (0, 1, m-1, m, m+k) and on both sides of the short-segment bound."""
import json
import os
import zlib
from collections import defaultdict

import numpy as np
import pytest

import oracle
from corpus import ASCII, DNA, mutate
from fuzzysearch_b200 import (_native, find_near_matches, find_near_matches_in_sequences,
                              has_near_match_in_sequences)
from parity import GOLDEN_DIR, assert_final_parity, load_golden, tup

pytestmark = pytest.mark.gpu

F = _native
BIG = 1 << 29
BOUND = F.FZB_SEG_SHORT_BYTES

# (name, pattern length, limits): one entry per route of fzb_search_segments
ROUTES = [
    ("exact", 10, dict(max_l_dist=0)),
    ("hamming-ngrams", 20, dict(max_substitutions=2, max_insertions=0, max_deletions=0)),
    ("hamming-lp", 5, dict(max_substitutions=2, max_insertions=0, max_deletions=0)),
    ("lev-ngrams-vm0", 20, dict(max_l_dist=2)),
    ("lev-ngrams-vm1", 60, dict(max_l_dist=3)),
    ("lev-ngrams-vm2", 80, dict(max_l_dist=2)),
    ("lev-lp", 6, dict(max_l_dist=2)),
    ("lev-lp-k>=m", 3, dict(max_l_dist=5)),
    ("generic-ngrams", 20, dict(max_substitutions=1, max_insertions=1, max_deletions=2, max_l_dist=2)),
    ("generic-lp", 7, dict(max_substitutions=1, max_insertions=1, max_deletions=2, max_l_dist=2)),
]


def _limits(kw):
    subs, ins, dels, l = oracle.normalize_params(kw.get("max_substitutions"), kw.get("max_insertions"),
                                                 kw.get("max_deletions"), kw.get("max_l_dist"))
    return tuple(BIG if x is None else min(x, BIG) for x in (subs, ins, dels)) + (l,)


def make_segments(seed, pat, alphabet, lengths, k):
    """Random segments of the given lengths with near-matches planted at the start, the middle and the end."""
    rng = np.random.default_rng(seed)
    alpha = np.frombuffer(alphabet, dtype=np.uint8)
    segs = []
    for n in lengths:
        s = bytearray(alpha[rng.integers(0, len(alpha), size=n)].tobytes())
        for where in ("start", "middle", "end"):
            v = mutate(rng, pat, alphabet, int(rng.integers(0, k + 2)))
            if len(v) == 0 or len(v) > n:
                continue
            pos = {"start": 0, "middle": (n - len(v)) // 2, "end": n - len(v)}[where]
            s[pos:pos + len(v)] = v
        segs.append(bytes(s))
    return segs


def search_segments(segs, pat, kw):
    blob = b"".join(segs)
    offsets = np.zeros(len(segs) + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum([len(s) for s in segs])
    hay = F.Haystack.from_host(blob if blob else b"\0")
    try:
        res = hay.search_segments(pat, offsets, *_limits(kw))
        out = {}
        for which in (F.RAW, F.FINAL):
            counts = res.segment_counts(which).tolist()
            s, e, d = res.arrays(which)
            rows = list(zip(s.tolist(), e.tolist(), d.tolist()))
            lists, pos = [], 0
            for c in counts:
                lists.append(rows[pos:pos + c])
                pos += c
            assert pos == len(rows)
            out[which] = lists
        stats = res.stats()
        res.close()
    finally:
        hay.close()
    return out[F.RAW], out[F.FINAL], stats


def check_against_oracle(segs, pat, kw, ctx=""):
    raw, fin, stats = search_segments(segs, pat, kw)
    assert len(raw) == len(fin) == len(segs)
    subs, ins, dels, l = _limits(kw)
    unconsolidated = l == 0 or (ins == 0 and dels == 0)
    for i, seg in enumerate(segs):
        ref_final, ref_raw = oracle.find_near_matches(pat, seg, return_raw=True, **kw)
        c = "%s segment %d (len %d)" % (ctx, i, len(seg))
        assert sorted(raw[i]) == sorted(tup(ref_raw)), c
        assert raw[i] == sorted(raw[i]), c  # (start, end, dist) order within a segment
        if unconsolidated:  # exact / Hamming: FINAL is the raw list
            assert fin[i] == tup(ref_final), c
        else:
            assert_final_parity(fin[i], ref_final, ref_raw, c)
    return stats


def seg_lengths(m, k, rng, long=True):
    out = [0, 1, max(m - 1, 0), m, m + k] + [int(x) for x in rng.integers(1, 400, size=6)]
    if long:
        out += [BOUND - 1, BOUND, BOUND + 1]
    return out


@pytest.mark.parametrize("route", [r[0] for r in ROUTES])
@pytest.mark.parametrize("alphabet", ["dna", "ascii"])
def test_segments_match_oracle_per_route(cuda_device, route, alphabet, long=True):
    name, m, kw = next(r for r in ROUTES if r[0] == route)
    alpha = DNA if alphabet == "dna" else ASCII
    rng = np.random.default_rng(zlib.crc32((route + alphabet).encode()))
    pat = bytes(np.frombuffer(alpha, np.uint8)[rng.integers(0, len(alpha), size=m)])
    k = _limits(kw)[3]
    segs = make_segments(int(rng.integers(1 << 30)), pat, alpha, seg_lengths(m, min(k, 8), rng, long), min(k, 4))
    check_against_oracle(segs, pat, kw, "%s/%s" % (route, alphabet))


def test_segments_are_isolated(cuda_device):
    """A pattern split across a seam, and near-matches that would need bytes of the neighbour (insertions running
    over the seam), are reported only as far as each segment alone allows."""
    pat = b"GATTACAGATTACA"
    segs = [pat[:7], pat[7:], b"TT" + pat[:-1], pat[1:] + b"CC", pat, b"", pat + pat[:5], pat[3:] + pat[:3]]
    for kw in (dict(max_l_dist=2), dict(max_l_dist=0), dict(max_substitutions=2, max_insertions=0, max_deletions=0),
               dict(max_substitutions=1, max_insertions=2, max_deletions=1, max_l_dist=2), dict(max_l_dist=4)):
        check_against_oracle(segs, pat, kw, repr(kw))
        got = find_near_matches_in_sequences(pat, segs, **kw)
        assert [[(x.start, x.end, x.dist) for x in lst] for lst in got] == \
            [[(x.start, x.end, x.dist) for x in find_near_matches(pat, s, **kw)] for s in segs]


def _golden_groups(records):
    groups = defaultdict(list)
    for rec in records:
        if rec["fn"] != "find_near_matches" or "exc" in rec:
            continue
        a = rec["args"]
        groups[(a[0], tuple(a[2:6]))].append((bytes.fromhex(a[1]), rec["result"]))
    return groups


def replay_golden(records, stride=1):
    groups = _golden_groups(records)
    n = 0
    for (phex, args), items in sorted(groups.items(), key=repr)[::stride]:
        pat = bytes.fromhex(phex)
        kw = dict(zip(("max_substitutions", "max_insertions", "max_deletions", "max_l_dist"), args))
        got = find_near_matches_in_sequences(pat, [h for h, _ in items], **kw)
        subs, ins, dels, l = oracle.normalize_params(*args)
        for (hay, result), ours in zip(items, got):
            ours = [(x.start, x.end, x.dist) for x in ours]
            ctx = "%s %r %s" % (phex, args, hay.hex())
            if l == 0 or (ins == 0 and dels == 0):
                assert ours == tup(result), ctx
            else:
                _, raw = oracle.find_near_matches(pat, hay, *args, return_raw=True)
                assert_final_parity(ours, result, raw, ctx)
            n += 1
    return n


def test_reference_fuzz_records_as_segmented_calls(cuda_device):
    """The find_near_matches records of tests/golden/ref_fuzz.json (outputs of the real reference), grouped by
    (pattern, limits), each group one segmented call."""
    assert replay_golden(load_golden("ref_fuzz.json")) >= 1400


def test_reference_short_reads_fixture(cuda_device, stride=1):
    """tests/golden/ref_segments.json: the real reference over seeded short reads with planted primers
    (tests/golden/gen_golden_segments.py); one segmented call per (primer, limits)."""
    with open(os.path.join(GOLDEN_DIR, "ref_segments.json")) as f:
        cases = json.load(f)["cases"]
    for case in cases[::stride]:
        pat = bytes.fromhex(case["pattern"])
        reads = [bytes.fromhex(r) for r in case["reads"]]
        got = find_near_matches_in_sequences(pat, reads, **case["kwargs"])
        subs, ins, dels, l = oracle.normalize_params(**case["kwargs"])
        for read, ours, ref in zip(reads, got, case["results"]):
            ours = [(x.start, x.end, x.dist) for x in ours]
            if l == 0 or (ins == 0 and dels == 0):
                assert ours == tup(ref)
            else:
                _, raw = oracle.find_near_matches(pat, read, return_raw=True, **case["kwargs"])
                assert_final_parity(ours, ref, raw, case["kwargs"])
        assert has_near_match_in_sequences(pat, reads, **case["kwargs"]) == [bool(r) for r in case["results"]]


def test_public_api_matches_the_per_item_loop(cuda_device):
    pat = b"ACGTTGCA"
    base = make_segments(7, pat, DNA, [30, 8, 0, 50, 7, 120], 2)
    text = [s.decode("latin-1") for s in base]
    variants = [base, [bytearray(s) for s in base], [memoryview(s) for s in base],
                [np.frombuffer(s, dtype=np.uint8) for s in base]]
    kws = [dict(max_l_dist=1), dict(max_l_dist=0), dict(max_substitutions=1, max_insertions=0, max_deletions=0),
           dict(max_substitutions=1, max_insertions=1, max_deletions=0, max_l_dist=1)]
    for kw in kws:
        for items in variants:
            got = find_near_matches_in_sequences(pat, items, **kw)
            exp = [find_near_matches(pat, s, **kw) for s in items]
            assert got == exp, kw
            for lst, e in zip(got, exp):
                for x, y in zip(lst, e):
                    assert type(x.matched) is type(y.matched) and x.matched == y.matched
            assert has_near_match_in_sequences(pat, items, **kw) == [bool(e) for e in exp]
        got = find_near_matches_in_sequences(pat.decode(), text, **kw)
        assert got == [find_near_matches(pat.decode(), s, **kw) for s in text]
        assert all(isinstance(x.matched, str) for lst in got for x in lst)
    # wide symbols and list items: the per-item loop (still on the device)
    wide = ["αβACGTα", "xxαβACG", ""]
    assert find_near_matches_in_sequences("αβACG", wide, max_l_dist=1) == \
        [find_near_matches("αβACG", s, max_l_dist=1) for s in wide]
    items = [[1, 2, 3, 4, 5], [9, 1, 2, 4, 5, 9]]
    assert find_near_matches_in_sequences([1, 2, 3, 4], items, max_l_dist=1) == \
        [find_near_matches([1, 2, 3, 4], s, max_l_dist=1) for s in items]
    # errors as find_near_matches raises them
    assert find_near_matches_in_sequences(pat, []) == []
    assert has_near_match_in_sequences(pat, [], max_l_dist=1) == []
    with pytest.raises(ValueError):
        find_near_matches_in_sequences(b"", base, max_l_dist=1)
    with pytest.raises(ValueError):
        find_near_matches_in_sequences(b"", base, max_l_dist=0)
    with pytest.raises(ValueError):
        find_near_matches_in_sequences(pat, base)
    with pytest.raises(TypeError):
        find_near_matches_in_sequences(pat, base, max_l_dist=-1)
    with pytest.raises(TypeError):
        find_near_matches_in_sequences(pat, base[:2] + ["ACGT"], max_l_dist=1)
    with pytest.raises(TypeError):
        find_near_matches_in_sequences(pat.decode(), text[:2] + [b"ACGT"], max_l_dist=1)


def test_launch_count_does_not_grow_with_the_number_of_segments(cuda_device, many=100000):
    pat = b"ACGTACGTTGCAACGTAC"
    rng = np.random.default_rng(3)
    for kw in (dict(max_l_dist=2), dict(max_substitutions=2, max_insertions=0, max_deletions=0)):
        launches = []
        for count in (10, many):
            lens = rng.integers(50, 200, size=count)
            alpha = np.frombuffer(DNA, np.uint8)
            segs = [alpha[rng.integers(0, 4, size=int(n))].tobytes() for n in lens]
            _, _, stats = search_segments(segs, pat, kw)
            assert stats["route"] == "segments"
            launches.append(stats["n_launches"])
        assert launches[0] == launches[1], launches


def test_refusals(cuda_device):
    hay = F.Haystack.from_host(b"ACGT" * 10)
    with pytest.raises(ValueError):
        hay.search_segments(b"ACG", [0, 50], BIG, BIG, BIG, 1)  # beyond the end
    with pytest.raises(ValueError):
        hay.search_segments(b"ACG", [0, 20, 10], BIG, BIG, BIG, 1)  # decreasing
    with pytest.raises(ValueError):
        hay.search_segments(b"ACG", [0, 20], BIG, BIG, BIG, 1, F.F_GLOBAL)
    hay.close()
    shard = F.Haystack.from_host(b"ACGT" * 10, global_len=80, own_lo=0, own_hi=40)
    with pytest.raises(ValueError):
        shard.search_segments(b"ACG", [0, 20], BIG, BIG, BIG, 1)
    shard.close()
