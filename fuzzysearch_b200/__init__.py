"""fuzzysearch_b200 -- B200-native (sm_100a CUDA) drop-in for fuzzysearch's near-match search.

Same public API as the reference (fuzzysearch/__init__.py:35-83):

>>> find_near_matches(b'PATTERN', b'---PATERN---', max_l_dist=1)
[Match(start=3, end=9, dist=1, matched=b'PATERN')]

Every search runs as hand-written CUDA kernels behind the C-ABI of libfuzzb200.so
(include/fuzzb200.h); there is no CPU fallback -- without the library or a GPU the calls raise.
"""
__version__ = "0.1.0"

__all__ = ["find_near_matches", "find_near_matches_batch", "find_near_matches_in_file", "find_near_matches_in_sequences",
           "has_near_match", "has_near_match_in_sequences", "Match", "LevenshteinSearchParams",
           "DeviceSequence", "ExactSearch", "SubstitutionsOnlySearch", "LevenshteinSearch",
           "GenericSearch", "choose_search_class", "search_exact"]

from .common import LevenshteinSearchParams, Match
from .search import (DeviceSequence, ExactSearch, GenericSearch, LevenshteinSearch,
                     SubstitutionsOnlySearch, search_exact)


def find_near_matches(subsequence, sequence, max_substitutions=None, max_insertions=None,
                      max_deletions=None, max_l_dist=None):
    """search for near-matches of subsequence in sequence (fuzzysearch/__init__.py:35-57).

    The nearly-matching parts of the sequence must meet the given limits on substitutions,
    insertions, deletions and their total (the Levenshtein distance)."""
    search_params = LevenshteinSearchParams(max_substitutions, max_insertions, max_deletions,
                                            max_l_dist)
    search_class = choose_search_class(search_params)
    matches = search_class.search(subsequence, sequence, search_params)
    return search_class.consolidate_matches(matches)


def has_near_match(subsequence, sequence, max_substitutions=None, max_insertions=None, max_deletions=None,
                   max_l_dist=None):
    """True iff find_near_matches(...) would return at least one match -- the public-API form of the
    reference's internal has_near_match_* helpers (substitutions_only.py:18-34,139-145,218-233;
    generic_search.py:240-253), with early termination: the sequence is searched in chunks of growing size and
    the call returns after the first chunk that holds a match (fzb_has_near_match)."""
    from .search import _lock_for, _prepare
    search_params = LevenshteinSearchParams(max_substitutions, max_insertions, max_deletions, max_l_dist)
    if len(subsequence) == 0:
        raise ValueError("Given subsequence is empty!")
    subs, ins, dels, l = search_params.unpacked
    big = 1 << 29
    subs, ins, dels = (big if subs is None else subs), (big if ins is None else ins), (big if dels is None else dels)
    with _lock_for(sequence):
        pat, hay, _, _ = _prepare(subsequence, sequence)
        return hay.has_near_match(pat, min(subs, big), min(ins, big), min(dels, big), l)


def find_near_matches_batch(subsequences, sequence, max_l_dist):
    """Many patterns over one sequence (uploaded once): -> list of find_near_matches(...) results.

    `max_l_dist` is one int or one per pattern.  Equivalent to
    ``[find_near_matches(p, sequence, max_l_dist=k) for p, k in zip(subsequences, ks)]``."""
    from . import _native
    subsequences = list(subsequences)
    ks = [max_l_dist] * len(subsequences) if isinstance(max_l_dist, int) else list(max_l_dist)
    if len(ks) != len(subsequences):
        raise ValueError("one max_l_dist per subsequence expected")
    for p, k in zip(subsequences, ks):
        LevenshteinSearchParams(None, None, None, k)  # same validation as find_near_matches
        if len(p) == 0:
            raise ValueError("Given subsequence is empty!")
    if not subsequences:
        return []
    from .search import AlphabetTooLarge, _lock_for, _prepare_many
    with _lock_for(sequence):
        try:
            pats, hay, slicer = _prepare_many(subsequences, sequence)
        except AlphabetTooLarge:
            # wide symbols and more than 255 distinct ones over all the patterns: no common byte alphabet,
            # so the patterns go one by one (each reduces the sequence to its own alphabet)
            return [find_near_matches(p, sequence, max_l_dist=k) for p, k in zip(subsequences, ks)]
        results, _ = hay.search_levenshtein_batch(pats, ks)
        out = []
        for res, k in zip(results, ks):
            # max_l_dist == 0 selects ExactSearch in find_near_matches (__init__.py:65-66), whose result is
            # the unconsolidated occurrence list (search_exact.py:80-89): the RAW stream of the k == 0 route
            s, e, d = res.arrays(_native.RAW if k == 0 else _native.FINAL)
            out.append([Match(a, b, c, matched=slicer(a, b)) for a, b, c in zip(s.tolist(), e.tolist(), d.tolist())])
            res.close()
    return out


def find_near_matches_in_sequences(subsequence, sequences, max_substitutions=None, max_insertions=None,
                                   max_deletions=None, max_l_dist=None):
    """One pattern over many sequences (reads, lines, records): -> one list of Match per sequence, equal to
    ``[find_near_matches(subsequence, s, ...) for s in sequences]`` (``Match.matched`` is a slice of that item).

    The items are packed into one buffer and searched in a single device pass (fzb_search_segments) instead of paying
    the fixed cost of a search per item.  Items may be bytes, bytearray, memoryview, numpy uint8 arrays or str; items
    with wide symbols, or list / tuple items, are searched one by one."""
    sequences = list(sequences)
    if not sequences:
        return []
    search_params = LevenshteinSearchParams(max_substitutions, max_insertions, max_deletions, max_l_dist)
    choose_search_class(search_params)
    from .search import search_sequences

    def per_item(s):
        return find_near_matches(subsequence, s, max_substitutions, max_insertions, max_deletions, max_l_dist)
    return search_sequences(subsequence, sequences, search_params, per_item)


def has_near_match_in_sequences(subsequence, sequences, max_substitutions=None, max_insertions=None,
                                max_deletions=None, max_l_dist=None):
    """-> one bool per sequence: True where find_near_matches_in_sequences(...) has a non-empty list (e.g. which reads
    contain the primer)."""
    sequences = list(sequences)
    if not sequences:
        return []
    search_params = LevenshteinSearchParams(max_substitutions, max_insertions, max_deletions, max_l_dist)
    from .search import search_sequences

    def per_item(s):
        return find_near_matches(subsequence, s, max_substitutions, max_insertions, max_deletions, max_l_dist)
    return search_sequences(subsequence, sequences, search_params, per_item, counts_only=True)


def choose_search_class(search_params):
    """fuzzysearch/__init__.py:60-83."""
    max_substitutions, max_insertions, max_deletions, max_l_dist = search_params.unpacked
    if max_l_dist == 0:
        return ExactSearch
    elif max_insertions == 0 and max_deletions == 0:
        return SubstitutionsOnlySearch
    elif max_l_dist <= min(
            (max_substitutions if max_substitutions is not None else (1 << 29)),
            (max_insertions if max_insertions is not None else (1 << 29)),
            (max_deletions if max_deletions is not None else (1 << 29)),
    ):
        return LevenshteinSearch
    else:
        return GenericSearch


def find_near_matches_in_file(subsequence, sequence_file, max_substitutions=None, max_insertions=None,
                              max_deletions=None, max_l_dist=None, _chunk_size=2 ** 20):
    """search for near-matches of subsequence in a file (fuzzysearch/__init__.py:86-200)."""
    from .file_search import find_near_matches_in_file as impl
    return impl(subsequence, sequence_file, max_substitutions, max_insertions, max_deletions,
                max_l_dist, _chunk_size)
