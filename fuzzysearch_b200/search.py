"""The four search classes -- the reference's plugin seam (SURVEY.md section 8b).

``fuzzysearch.choose_search_class`` (__init__.py:60-83) picks one of ExactSearch /
SubstitutionsOnlySearch / LevenshteinSearch / GenericSearch, each a ``FuzzySearchBase`` with
``search(subsequence, sequence, search_params)`` and ``consolidate_matches(matches)``
(common.py:192-209).  Here each ``search`` is ONE call into libfuzzb200.so (sm_100a kernels);
there is no CPU implementation behind them.
"""
import threading
from collections.abc import Sequence

import numpy as np

from . import _native
from .common import FuzzySearchBase, Match, consolidate_overlapping_matches

try:  # optional, exactly like the reference (search_exact.py:14-19): Bio.Seq.Seq sequences are text
    from Bio.Seq import Seq as _BioSeq
except ImportError:
    _BioSeq = None


def _text(seq):
    """Bio.Seq.Seq -> its str (the reference walks a Seq with Seq.find / item access, i.e. as text); anything
    else unchanged.  ``Match.matched`` is still sliced from the ORIGINAL object."""
    if _BioSeq is not None and isinstance(seq, _BioSeq):
        return str(seq)
    return seq


__all__ = ["DeviceSequence", "ExactSearch", "SubstitutionsOnlySearch", "LevenshteinSearch",
           "GenericSearch", "RawMatches", "search_exact", "search_sequences"]


class DeviceSequence(object):
    """A haystack kept resident in HBM so that several searches reuse one upload.

    ``find_near_matches(pattern, DeviceSequence(data), ...)`` behaves like
    ``find_near_matches(pattern, data, ...)``.  Byte-like data and latin-1 encodable ``str`` are uploaded
    once; a general-Unicode ``str`` (or a list / tuple of hashable items) is reduced to bytes relative to the
    PATTERN's alphabet (see ``_reduce``), so it is uploaded again whenever a search brings a pattern with a
    different set of symbols."""

    def __init__(self, data=None, device=0, _haystack=None, _host=None):
        # held across bind (re-reduction to a new pattern alphabet) + search + copy-out of the consolidated list:
        # threads sharing one resident sequence take turns, like callers of the reference under the GIL
        self._lock = threading.RLock()
        self._wide = None        # the original str / list / tuple when the byte form depends on the pattern
        self._alphabet = None    # ... and the pattern alphabet the resident bytes were reduced with
        self._is_str = False
        self._kind = "bytes"
        self._orig = None        # a Bio.Seq.Seq: `matched` is sliced from it
        if _haystack is not None:
            self.haystack, self._host = _haystack, _host
            return
        if _text(data) is not data:
            self._orig, data = data, _text(data)
        self._kind = _kind(data)
        self._is_str = self._kind == "str"
        host = _narrow(data, self._kind)
        if host is not None:
            self._host = host
            self.haystack = _native.Haystack.from_host(host, device=device)
        else:
            self._host = None
            self._wide = data
            self.haystack = _native.Haystack.alloc(max(len(data), 1), device=device)

    def __len__(self):
        if self._orig is not None:
            return len(self._orig)
        return len(self._wide) if self._wide is not None else len(self.haystack)

    def _bind(self, subsequence):
        """-> the pattern as bytes in this sequence's byte alphabet (re-reducing the sequence if needed)."""
        return self._bind_many([subsequence])[0]

    def _bind_many(self, subsequences):
        subsequences = [_text(p) for p in subsequences]
        kinds = set(_kind(p) for p in subsequences)
        if kinds != {self._kind}:
            raise TypeError("subsequence and sequence must both be str or both be byte-like")
        if self._wide is None:
            pats = [_narrow(p, self._kind) for p in subsequences]
            if all(p is not None for p in pats):
                return pats
            # a pattern with symbols outside latin-1 over a latin-1 sequence: those symbols match nothing,
            # but the search still has to run with them in place -- reduce both sides
            self._wide = self.slice(0, len(self))
        alphabet = _make_alphabet(subsequences, self._kind)
        if alphabet != self._alphabet:
            _upload_reduced(self.haystack, self._wide, self._kind, alphabet)
            self._alphabet = alphabet
        return [_rename(p, self._kind, alphabet) for p in subsequences]

    def slice(self, start, end):
        if self._orig is not None:
            return self._orig[start:end]
        if self._wide is not None:
            return self._wide[start:end]
        if self._host is not None:
            b = bytes(memoryview(self._host)[start:end])
        else:
            b = self.haystack.read(start, end - start)
        return b.decode("latin-1") if self._is_str else b

    def close(self):
        self.haystack.close()


def _kind(seq):
    """'str' | 'items' (list / tuple of hashable items) | 'bytes' (anything byte-like)"""
    if isinstance(seq, str):
        return "str"
    if isinstance(seq, (list, tuple)):
        return "items"
    return "bytes"


def _narrow(seq, kind):
    """-> uint8 view when `seq` has single-byte symbols of its own (byte-like: zero-copy; latin-1 encodable
    str: encoded), else None."""
    if kind == "str":
        try:
            return np.frombuffer(seq.encode("latin-1"), dtype=np.uint8)
        except UnicodeEncodeError:
            return None
    if kind == "items":
        return None
    return _native.as_u8(seq)


def _coerce(seq):
    """-> (uint8 view, is_str) for sequences with single-byte symbols."""
    kind = _kind(seq)
    a = _narrow(seq, kind)
    if a is None:
        raise TypeError("a sequence of single-byte symbols is required here (got %s)" % type(seq).__name__)
    return a, kind == "str"


class AlphabetTooLarge(_native.UnsupportedError):
    pass


def _make_alphabet(subsequences, kind):
    """The reduction every algorithm on the path is invariant under (they only ever compare a pattern symbol
    with a sequence symbol -- levenshtein_ngram.py:49,113, levenshtein.py:83, generic_search.py:86,
    substitutions_only.py:93-99, search_exact.py:45-56): pattern symbol -> 1 + its rank among the distinct
    symbols of the pattern(s), any other sequence symbol -> 0.

    str: the sorted code points (the device reduces the sequence side, k_reduce_symbols);
    items: {item: byte} (Python objects can only be numbered by the interpreter)."""
    if kind == "str":
        alphabet = sorted(set(ord(c) for p in subsequences for c in p))
        if len(alphabet) > _native.FZB_MAX_PATTERN:
            raise AlphabetTooLarge("more than %d distinct pattern symbols" % _native.FZB_MAX_PATTERN)
        return alphabet
    ids = {}
    for p in subsequences:
        for item in p:
            if item not in ids:
                if len(ids) == _native.FZB_MAX_PATTERN:
                    raise AlphabetTooLarge("more than %d distinct pattern symbols" % _native.FZB_MAX_PATTERN)
                ids[item] = len(ids) + 1
    return ids


def _rename(subsequence, kind, alphabet):
    if kind == "str":
        rank = {c: i + 1 for i, c in enumerate(alphabet)}
        return np.fromiter((rank[ord(c)] for c in subsequence), dtype=np.uint8, count=len(subsequence))
    return np.fromiter((alphabet[x] for x in subsequence), dtype=np.uint8, count=len(subsequence))


def _code_units(text):
    """str -> its code units as a numpy array: UCS-2 (uint16) when every character is in the BMP, else
    UTF-32 (uint32).  Lone surrogates are symbols like any other ('surrogatepass')."""
    if not text or max(text) < "\U00010000":
        return np.frombuffer(text.encode("utf-16-le", "surrogatepass"), dtype=np.uint16)
    return np.frombuffer(text.encode("utf-32-le", "surrogatepass"), dtype=np.uint32)


def _upload_reduced(hay, sequence, kind, alphabet):
    if kind == "str":
        hay.upload_symbols(_code_units(sequence), alphabet)
    else:
        get = alphabet.get
        try:
            hay.upload(np.fromiter((get(x, 0) for x in sequence), dtype=np.uint8, count=len(sequence)))
        except TypeError:
            raise TypeError("sequence items must be hashable")


class RawMatches(Sequence):
    """The raw match stream of one search, materialised LAZILY: ``find_near_matches`` only needs the
    consolidated list (``.final``, built from the device-side consolidation), so the raw ``Match``
    objects -- one Python object and one slice per raw record -- are only built if somebody iterates,
    indexes or compares this object (the search-class ``search()`` contract of the reference,
    common.py:192-197, is "an iterable of Match")."""

    def __init__(self, result, slicer, consolidated):
        self._result = result
        self._slicer = slicer
        self._list = None
        self.stats = result.stats()
        self.final = _to_matches(result, _native.FINAL, slicer) if consolidated else None
        self._n = result.count(_native.RAW)

    def materialize(self):
        if self._list is None:
            self._list = _to_matches(self._result, _native.RAW, self._slicer)
            self._result.close()
            self._result = None
        return self._list

    def __len__(self):
        return self._n

    def __iter__(self):
        return iter(self.materialize())

    def __getitem__(self, i):
        return self.materialize()[i]

    def __eq__(self, other):
        if isinstance(other, RawMatches):
            other = other.materialize()
        return self.materialize() == other

    def __ne__(self, other):
        return not self.__eq__(other)

    __hash__ = None

    def __repr__(self):
        return repr(self.materialize())

    def __del__(self):
        if getattr(self, "_result", None) is not None:
            self._result.close()


def _prepare(subsequence, sequence):
    """-> (pattern u8, haystack handle, slicer, owns_handle)"""
    pats, hay, slicer = _prepare_many([subsequence], sequence)
    return pats[0], hay, slicer, False


def _prepare_many(subsequences, sequence):
    """-> (patterns as u8 arrays, haystack handle holding the sequence, slicer)"""
    if isinstance(sequence, DeviceSequence):
        return sequence._bind_many(subsequences), sequence.haystack, sequence.slice
    original, sequence = sequence, _text(sequence)
    subsequences = [_text(p) for p in subsequences]
    kind = _kind(sequence)
    if any(_kind(p) != kind for p in subsequences):
        raise TypeError("subsequence and sequence must both be str or both be byte-like")
    pats = [_narrow(p, kind) for p in subsequences]
    host = _narrow(sequence, kind) if all(p is not None for p in pats) else None
    if host is not None:
        hay = _workspace(host.size)
        hay.upload(host)
    else:  # wide symbols on either side: reduce both to the patterns' alphabet
        alphabet = _make_alphabet(subsequences, kind)
        pats = [_rename(p, kind, alphabet) for p in subsequences]
        hay = _workspace(len(sequence))
        _upload_reduced(hay, sequence, kind, alphabet)
    if kind != "bytes" or isinstance(sequence, (bytes, bytearray)):
        def slicer(s, e):
            return original[s:e]
    else:
        mv = memoryview(host)

        def slicer(s, e):
            return bytes(mv[s:e])
    return pats, hay, slicer


_WORKSPACE = {}
# One lock per process around upload + search + copy-out of the SHARED workspace: ctypes drops the GIL
# during the native calls, so without it two threads calling find_near_matches() would overwrite each
# other's haystack mid-search.  (The reference is serialised by the GIL.)  A DeviceSequence has its own lock
# (and the library serialises the calls on one handle), so searches of different resident sequences overlap.
_WORKSPACE_LOCK = threading.RLock()


def _lock_for(sequence):
    return sequence._lock if isinstance(sequence, DeviceSequence) else _WORKSPACE_LOCK


def _workspace(nbytes, device=0):
    """A cached device buffer for plain (host) sequences: like the reference's reusable chunk buffer
    (__init__.py:141-145), a search then costs one H2D copy instead of allocations."""
    ws = _WORKSPACE.get(device)
    if ws is None or ws[1] < nbytes:
        if ws is not None:
            ws[0].close()
        cap = max(nbytes + nbytes // 8, 1 << 20)
        ws = (_native.Haystack.alloc(cap, device=device), cap)
        _WORKSPACE[device] = ws
    return ws[0]


def release_workspace():
    for ws in _WORKSPACE.values():
        ws[0].close()
    _WORKSPACE.clear()
    _native.lib().fzb_release_workspace()


def _to_matches(result, which, slicer):
    s, e, d = result.arrays(which)
    return [Match(a, b, c, matched=slicer(a, b)) for a, b, c in zip(s.tolist(), e.tolist(), d.tolist())]


def _run(subsequence, sequence, call, consolidated):
    with _lock_for(sequence):
        pat, hay, slicer, _ = _prepare(subsequence, sequence)
        res = call(hay, pat)
        try:
            return RawMatches(res, slicer, consolidated)
        except BaseException:
            res.close()
            raise


def search_exact(subsequence, sequence, start_index=0, end_index=None):
    """fuzzysearch.search_exact.search_exact (search_exact.py:22-56): the start indexes of the (overlapping)
    occurrences of `subsequence` lying wholly inside ``sequence[start_index:end_index]``, ascending.

    Only the window travels to / is scanned on the device: a host sequence is sliced before the upload, a
    ``DeviceSequence`` is searched through a view of its resident buffer (fzb_search_exact_window)."""
    if len(subsequence) == 0:
        raise ValueError("subsequence must not be empty")
    sequence = _text(sequence)  # a Bio.Seq.Seq is searched as its text; the result is positions only
    n = len(sequence)
    if end_index is None:
        end_index = n
    start_index = max(0, min(start_index, n))               # clamp(...) search_exact.py:29-30
    end_index = max(start_index, min(end_index, n))
    if isinstance(sequence, DeviceSequence):
        with sequence._lock:
            pat = sequence._bind(subsequence)
            res = sequence.haystack.search_exact(pat, start=start_index, end=end_index)
            starts = res.arrays(_native.RAW)[0]  # positions are already those of the whole sequence
            res.close()
        return starts.tolist()
    else:
        if _kind(sequence) == "bytes" and not isinstance(sequence, (bytes, bytearray)):
            window = memoryview(_native.as_u8(sequence))[start_index:end_index]
        elif start_index == 0 and end_index == n:
            window = sequence
        else:
            window = sequence[start_index:end_index]
        with _WORKSPACE_LOCK:
            pat, hay, _, _ = _prepare(subsequence, window)
            res = hay.search_exact(pat)
            starts = res.arrays(_native.RAW)[0]
            res.close()
        return (starts + start_index).tolist() if start_index else starts.tolist()


class ExactSearch(FuzzySearchBase):
    """search_exact.py:80-89."""

    @classmethod
    def search(cls, subsequence, sequence, search_params=None):
        if len(subsequence) == 0:
            raise ValueError("subsequence must not be empty")
        return _run(subsequence, sequence, lambda h, p: h.search_exact(p), False)

    @classmethod
    def extra_items_for_chunked_search(cls, subsequence, search_params):
        return 0


class SubstitutionsOnlySearch(FuzzySearchBase):
    """substitutions_only.py:288-301."""

    @classmethod
    def search(cls, subsequence, sequence, search_params):
        if len(subsequence) == 0:
            raise ValueError("Given subsequence is empty!")
        actual_max_subs = min(x for x in [search_params.max_l_dist, search_params.max_substitutions]
                              if x is not None)
        return _run(subsequence, sequence, lambda h, p: h.search_hamming(p, actual_max_subs), False)

    @classmethod
    def extra_items_for_chunked_search(cls, subsequence, search_params):
        return 0


class LevenshteinSearch(FuzzySearchBase):
    """levenshtein.py:151-164."""

    @classmethod
    def search(cls, subsequence, sequence, search_params):
        if len(subsequence) == 0:
            raise ValueError("Given subsequence is empty!")
        k = search_params.max_l_dist
        return _run(subsequence, sequence, lambda h, p: h.search_levenshtein(p, k), True)

    @classmethod
    def consolidate_matches(cls, matches):
        return consolidate_overlapping_matches(matches)

    @classmethod
    def extra_items_for_chunked_search(cls, subsequence, search_params):
        return search_params.max_l_dist


class GenericSearch(FuzzySearchBase):
    """generic_search.py:256-273."""

    @classmethod
    def search(cls, subsequence, sequence, search_params):
        if len(subsequence) == 0:
            raise ValueError("Given subsequence is empty!")
        subs, ins, dels, l = search_params.unpacked
        return _run(subsequence, sequence, lambda h, p: h.search_generic(p, subs, ins, dels, l), True)

    @classmethod
    def consolidate_matches(cls, matches):
        return consolidate_overlapping_matches(matches)

    @classmethod
    def extra_items_for_chunked_search(cls, subsequence, search_params):
        return max(x for x in [search_params.max_l_dist, search_params.max_insertions] if x is not None)


def _pack_sequences(subsequence, sequences):
    """-> (pattern u8, packed bytes, offsets uint64[n + 1], slicers) when the pattern and every item have single-byte
    symbols of one kind, else None (wide symbols or list / tuple items: no byte alphabet shared by all the items).
    Raises the TypeError find_near_matches raises for an item of the other kind."""
    pattern = _text(subsequence)
    kind = _kind(pattern)
    if kind == "items" or any(isinstance(s, DeviceSequence) for s in sequences):
        return None
    pat = _narrow(pattern, kind)
    parts, slicers = [], []
    for original in sequences:
        seq = _text(original)
        if _kind(seq) != kind:
            raise TypeError("subsequence and sequence must both be str or both be byte-like")
        if kind == "str" or isinstance(seq, (bytes, bytearray)):
            part = seq.encode("latin-1") if kind == "str" and pat is not None else seq
            parts.append(part)
            slicers.append(original)
        else:
            host = _native.as_u8(seq)
            parts.append(host)
            slicers.append(memoryview(host))
    if pat is None:
        return None
    lengths = np.fromiter((len(x) for x in parts), dtype=np.uint64, count=len(parts))
    blob = b"".join(parts)
    offsets = np.zeros(len(parts) + 1, dtype=np.uint64)
    np.cumsum(lengths, out=offsets[1:])
    return pat, blob, offsets, slicers


def search_sequences(subsequence, sequences, search_params, per_item, counts_only=False):
    """find_near_matches of one pattern in each of `sequences` through fzb_search_segments: one upload of all the items
    packed back to back and one native call per FZB_SEG_MAX_COUNT items (the segment number's bits in a raw record).
    -> one list of Match per item (counts_only: one bool per item, true where that list is non-empty).

    `per_item(sequence)` is the fallback when no byte alphabet is shared by all the items (wide symbols, list / tuple
    items, resident DeviceSequence items): the items then go one by one, as find_near_matches_batch does."""
    subs, ins, dels, l = search_params.unpacked
    if len(subsequence) == 0:
        raise ValueError("subsequence must not be empty" if l == 0 else "Given subsequence is empty!")
    try:
        packed = _pack_sequences(subsequence, sequences)
    except UnicodeEncodeError:  # a str item outside latin-1
        packed = None
    if packed is None:
        return [bool(per_item(s)) if counts_only else per_item(s) for s in sequences]
    pat, blob, offsets, slicers = packed
    big = 1 << 29
    subs, ins, dels = (big if subs is None else min(subs, big)), (big if ins is None else min(ins, big)), \
        (big if dels is None else min(dels, big))
    n_items = len(slicers)
    out = []
    with _WORKSPACE_LOCK:
        hay = _workspace(len(blob))
        hay.upload(np.frombuffer(blob, dtype=np.uint8))
        for lo in range(0, n_items, _native.FZB_SEG_MAX_COUNT):
            hi = min(n_items, lo + _native.FZB_SEG_MAX_COUNT)
            res = hay.search_segments(pat, offsets[lo:hi + 1], subs, ins, dels, l)
            try:
                counts = res.segment_counts(_native.FINAL).tolist()
                if counts_only:
                    out.extend(c > 0 for c in counts)
                    continue
                starts, ends, dists = (a.tolist() for a in res.arrays(_native.FINAL))
            finally:
                res.close()
            pos = 0
            for i, c in enumerate(counts):
                if not c:
                    out.append([])
                    continue
                src = slicers[lo + i]
                if isinstance(src, memoryview):
                    out.append([Match(a, b, d, matched=bytes(src[a:b]))
                                for a, b, d in zip(starts[pos:pos + c], ends[pos:pos + c], dists[pos:pos + c])])
                else:
                    out.append([Match(a, b, d, matched=src[a:b])
                                for a, b, d in zip(starts[pos:pos + c], ends[pos:pos + c], dists[pos:pos + c])])
                pos += c
    return out
