/*
 * fuzzb200.h -- C-ABI of libfuzzb200.so: the B200-native (sm_100a) replacement for the
 * fuzzysearch hot path (bounded-Levenshtein / Hamming / generic near-match search of a short
 * byte pattern in a long byte haystack).
 *
 * Boundary.  In the reference the hot path sits behind the four search classes selected by
 * fuzzysearch.choose_search_class (src/fuzzysearch/__init__.py:60-83) -- ExactSearch,
 * SubstitutionsOnlySearch, LevenshteinSearch, GenericSearch -- each a FuzzySearchBase
 * (src/fuzzysearch/common.py:192-209) with search(subsequence, sequence, search_params) and
 * consolidate_matches(matches).  The reference's own native seams (search_exact_byteslike,
 * _common.c:5-112; c_expand_short/long, _levenshtein_ngrams.pyx:9-154;
 * substitutions_only_find_near_matches_ngrams_byteslike, _substitutions_only.c:4-50;
 * c_find_near_matches_generic_linear_programming, _generic_search.pyx:25-56) are per-candidate /
 * per-pass calls -- the wrong granularity for a GPU -- so each entry point below replaces one whole
 * search-class call instead.  INTEGRATION.md shows the ctypes stub that binds them.
 *
 * Conventions: every function returns 0 on success or a negative FZB_E_* code; the message is
 * available from fzb_last_error() (thread-local).  No C++ exceptions, Python objects or torch types
 * cross the ABI.  The caller owns every input buffer (copied during the call, never retained) and
 * every handle (explicit destroy).  Distinct handles may be used from distinct threads concurrently;
 * calls on one handle are serialised inside the library (per-handle mutex).
 *
 * Semantics are bit-exact with the reference's PURE-PYTHON path (SURVEY.md F6/F7): raw match
 * streams are element-for-element those of the cited generators; the consolidated list follows
 * consolidate_overlapping_matches (common.py:185-189) with ties inside a group (which the reference
 * leaves to set-iteration order) broken towards the smallest (start, end).
 */
#ifndef FUZZB200_H
#define FUZZB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default) /* the library is built with -fvisibility=hidden */
#endif

#define FZB_VERSION 100 /* 0.1.0 */

/* error codes */
#define FZB_OK 0
#define FZB_E_INVALID (-1)     /* bad argument (reference raises ValueError/TypeError) */
#define FZB_E_CUDA (-2)        /* CUDA runtime failure (no device, OOM, launch error) */
#define FZB_E_UNSUPPORTED (-3) /* valid for the reference but outside this library's limits */
#define FZB_E_NGRAM_ZERO (-4)  /* "the subsequence length must be greater than max_l_dist" */

#define FZB_MAX_PATTERN 255 /* bytes */

/* which result list */
#define FZB_RAW 0   /* the raw match stream, reference generation order */
#define FZB_FINAL 1 /* after the search class's consolidate_matches() */

/* fzb_search_* flags */
#define FZB_F_NO_FINAL 1u     /* skip consolidation (raw stream only) */
#define FZB_F_FORCE_DENSE 2u  /* force the every-position candidate filter (testing) */
#define FZB_F_FORCE_LP 4u     /* Levenshtein/generic: force the "linear programming" route */
#define FZB_F_FORCE_NGRAMS 8u /* Levenshtein/generic/Hamming: force the n-gram route */
#define FZB_F_TINY_LIST 16u   /* testing: cap the granule work list and the hit list at 8 entries (overflow paths) */
#define FZB_F_FORCE_SAMPLED 64u /* testing: use the sampled filter whenever its lemma holds, even if the
                                 byte statistics say it is not selective */
#define FZB_F_GLOBAL 32u      /* multi-GPU: FINAL becomes the GLOBAL consolidated list of all shards: every rank
                                 stores its groups into every other rank's receive area over NVLink peer
                                 memory and merges the seams on the device, on the search's own stream, right
                                 behind the kernels (needs fzb_haystack_comm_init / fzb_comm_init_local on every
                                 rank; collective: every rank must issue the same searches in the same order) */

struct fzb_stats_s;
typedef struct fzb_haystack fzb_haystack; /* a device-resident sequence (or one shard of it) */
typedef struct fzb_result fzb_result;     /* the matches of one search */

int fzb_version(void);
/* number of usable CUDA devices (0 if none / driver missing); never fails */
int fzb_device_count(void);
const char *fzb_last_error(void);

/* Upload `n` bytes of host memory to `device` as a whole sequence [0, n). */
int fzb_haystack_create(const uint8_t *host, uint64_t n, int device, fzb_haystack **out);

/*
 * Multi-GPU shard (SURVEY.md section 8e): the global sequence has `global_len` bytes; this handle
 * holds bytes [buf_lo, buf_lo + buf_len) of it (`host` points at byte buf_lo) and OWNS the matches
 * whose anchor (n-gram hit index / Hamming start / LP start) lies in [own_lo, own_hi).  The caller
 * must supply a halo: buf_lo <= max(0, own_lo - halo) and buf_lo + buf_len >= min(global_len,
 * own_hi + halo) with halo = len(pattern) + max_l_dist of the searches to be run (checked per
 * search).  Window clipping rules of the reference apply at 0 and global_len only, never at shard
 * seams, so the union of the shards' raw streams equals the single-device raw stream.
 */
int fzb_haystack_create_shard(const uint8_t *host, uint64_t buf_len, uint64_t buf_lo,
                              uint64_t global_len, uint64_t own_lo, uint64_t own_hi, int device,
                              fzb_haystack **out);

/* Adopt an existing device allocation (not freed by destroy).  `dev_ptr` must be 16-byte aligned
 * and readable for buf_len rounded up to a multiple of 128 bytes plus 128. Used by bench.py to scan
 * corpora generated on the device. */
int fzb_haystack_adopt_device(const void *dev_ptr, uint64_t buf_len, uint64_t buf_lo,
                              uint64_t global_len, uint64_t own_lo, uint64_t own_hi, int device,
                              fzb_haystack **out);

/* Allocate an uninitialised device-resident shard (same geometry arguments as
 * fzb_haystack_create_shard; a whole sequence is buf_lo = own_lo = 0, buf_len = global_len = own_hi)
 * and return its device pointer, for callers that fill it on the device. */
int fzb_haystack_alloc(uint64_t buf_len, uint64_t buf_lo, uint64_t global_len, uint64_t own_lo,
                       uint64_t own_hi, int device, fzb_haystack **out, void **dev_ptr);

/* Fill an fzb_haystack_alloc'ed sequence with a seeded synthetic corpus ON THE DEVICE: byte i =
 * alphabet[hash64(seed, i) % alphabet_len] (counter-based, so any shard of the global sequence can
 * be generated independently); host code can reproduce any slice with fzb_synth_host. */
int fzb_haystack_fill_synthetic(fzb_haystack *h, const uint8_t *alphabet, uint32_t alphabet_len,
                                uint64_t seed);
void fzb_synth_host(uint8_t *dst, uint64_t global_offset, uint64_t n, const uint8_t *alphabet,
                    uint32_t alphabet_len, uint64_t seed);
/* Overwrite bytes [global_offset, global_offset+n) of the sequence (must lie inside the buffer). */
int fzb_haystack_write(fzb_haystack *h, uint64_t global_offset, const uint8_t *src, uint64_t n);
/* Read bytes back (for Match.matched and tests). */
int fzb_haystack_read(fzb_haystack *h, uint64_t global_offset, uint8_t *dst, uint64_t n);

/* NCCL plumbing for FZB_F_GLOBAL (one process per GPU).  Rank 0 obtains a unique id and ships it to
 * the other ranks by any means (fuzzysearch_b200/sharding.py: a plain TCP rendezvous); then every rank calls
 * fzb_haystack_comm_init with its shard handle (collective, blocking).  libnccl.so.2 is resolved at
 * run time (dlopen), so the library has no link-time NCCL dependency. */
#define FZB_NCCL_ID_BYTES 128
/* Optional, before the first NCCL use: load this libnccl.so.2 instead of the default search path.  A
 * process that will also import torch must load torch's bundled NCCL (the same SONAME is shared), which
 * the Python binding arranges automatically. */
void fzb_nccl_set_library(const char *path);
int fzb_nccl_unique_id(uint8_t id[FZB_NCCL_ID_BYTES]);
int fzb_haystack_comm_init(fzb_haystack *h, const uint8_t id[FZB_NCCL_ID_BYTES], int rank, int world_size);
/* The same world inside ONE process: handles[r] becomes rank r of world_size shards (on one GPU or on several
 * GPUs with peer access).  No NCCL: the shards reach each other's receive areas directly.  FZB_F_GLOBAL searches
 * must then be issued on all handles CONCURRENTLY (one thread per handle): each one waits on the device for the
 * others' groups (bounded by a timeout).  Used by the tests to run the multi-rank reduction on a single GPU. */
int fzb_comm_init_local(fzb_haystack **handles, int world_size);
/* The multi-process world without NCCL: every rank calls fzb_p2p_export (allocates its receive area, returns its CUDA
 * IPC handle), the caller all-gathers the handles by any means (rank-major, FZB_IPC_HANDLE_BYTES each), every rank
 * calls fzb_p2p_connect; if any rank failed, all call fzb_p2p_disable.  Works for processes on different GPUs of a node
 * AND for processes sharing one GPU.  No staged fallback in such a world (a shard with more groups than a slot holds
 * makes the search fail with FZB_E_UNSUPPORTED on every rank). */
#define FZB_IPC_HANDLE_BYTES 64
int fzb_p2p_export(fzb_haystack *h, int rank, int world_size, uint8_t handle[FZB_IPC_HANDLE_BYTES]);
int fzb_p2p_connect(fzb_haystack *h, const uint8_t *handles);
void fzb_p2p_disable(fzb_haystack *h);
/* 1 if FZB_F_GLOBAL searches on this handle reduce over peer memory (k_push / k_merge), 0 if they take the
 * staged NCCL + host path (CUDA IPC or peer access unavailable). */
int fzb_haystack_p2p_enabled(const fzb_haystack *h);

/* Replace the contents of a whole-sequence handle with `n` new host bytes (n <= the capacity the
 * handle was created with); the device allocations are reused -- the analogue of the reference's
 * reusable chunk buffer in _search_binary_file (__init__.py:141-171). */
int fzb_haystack_upload(fzb_haystack *h, const uint8_t *host, uint64_t n);

/* The same for a sequence of WIDE symbols -- a general-Unicode str as UTF-32 (width 4) or UCS-2 (width 2)
 * code units, or any sequence whose items the caller has numbered -- which the reference searches through
 * str.find / list.index (search_exact.py:11-19,32-51) and per-item `!=` (levenshtein_ngram.py:49,113).
 * Every algorithm on the path only ever compares a pattern symbol with a sequence symbol, so the sequence is
 * reduced ON THE DEVICE to one byte per symbol: `alphabet` = the pattern's distinct symbols, strictly
 * ascending, n_alpha <= FZB_MAX_PATTERN; symbol alphabet[i] becomes byte i+1 and every other symbol byte 0.
 * Search it with the pattern renamed the same way (pattern byte = 1 + rank of the symbol in `alphabet`);
 * positions in the results are symbol indexes.  The handle must be a whole (unsharded) sequence. */
int fzb_haystack_upload_symbols(fzb_haystack *h, const void *host, uint64_t n, uint32_t width,
                                const uint32_t *alphabet, uint32_t n_alpha);

/* Page-locked host memory for fast host<->device copies (cudaHostAlloc); NULL on failure. */
void *fzb_host_alloc(uint64_t n);
void fzb_host_free(void *p);

/* Device-side stopwatch on the handle's stream: start records a CUDA event, stop records another,
 * waits for it and returns the elapsed milliseconds (covers every kernel and copy the handle
 * enqueued in between, including idle gaps). */
int fzb_timer_start(fzb_haystack *h);
int fzb_timer_stop(fzb_haystack *h, double *ms);

uint64_t fzb_haystack_len(const fzb_haystack *h); /* global length */
void fzb_haystack_destroy(fzb_haystack *h);

/*
 * LevenshteinSearch.search (levenshtein.py:151-156 -> find_near_matches_levenshtein :9-38):
 * k == 0 exact; len(pattern)//(k+1) >= 3 the n-gram search (levenshtein_ngram.py:159-198);
 * else the "linear programming" NFA (levenshtein.py:52-148).  FINAL =
 * consolidate_overlapping_matches.
 */
int fzb_search_levenshtein(fzb_haystack *h, const uint8_t *pattern, uint32_t m, uint32_t max_l_dist,
                           uint32_t flags, fzb_result **out);

/*
 * SubstitutionsOnlySearch.search (substitutions_only.py:288-297 ->
 * find_near_matches_substitutions :37-63): every start p in [0, n-m] with
 * Hamming(pattern, H[p:p+m]) <= max_subs, ascending, dist = exact Hamming distance.
 * FINAL == RAW (consolidate_matches is the base no-op, common.py:198-205).
 */
int fzb_search_hamming(fzb_haystack *h, const uint8_t *pattern, uint32_t m, uint32_t max_subs,
                       uint32_t flags, fzb_result **out);

/*
 * GenericSearch.search (generic_search.py:256-261 -> find_near_matches_generic :25-54) with the
 * normalised limits of LevenshteinSearchParams (common.py:100-116).
 */
int fzb_search_generic(fzb_haystack *h, const uint8_t *pattern, uint32_t m, uint32_t max_subs,
                       uint32_t max_ins, uint32_t max_dels, uint32_t max_l_dist, uint32_t flags,
                       fzb_result **out);

/*
 * Batch of Levenshtein searches over ONE resident haystack (BASELINE.json configs[4]): `count` patterns
 * concatenated in `patterns` (pattern i = patterns[offsets[i] : offsets[i+1]]), each with its own
 * max_l_dist[i].  out[i] receives an ordinary fzb_result for pattern i (the caller destroys each).
 * The patterns share passes over the haystack (DESIGN.md section 5.5): ONE scan for every pattern the
 * q-sample lemma covers, ONE for the other n-gram-route patterns, ONE per 64 LP-route patterns; patterns
 * longer than 64 bytes are searched one by one.  Each out[i] is exactly what fzb_search_levenshtein would
 * return for pattern i.  `total` (optional) sums the statistics.  On error nothing is returned.
 */
int fzb_search_levenshtein_batch(fzb_haystack *h, const uint8_t *patterns, const uint32_t *offsets,
                                 const uint32_t *max_l_dist, uint32_t count, uint32_t flags,
                                 fzb_result **out, struct fzb_stats_s *total);

/*
 * One pattern over MANY sequences in one device pass: the segments [offsets[i], offsets[i+1]) (i < count) of the
 * whole-sequence handle `h` (offsets non-decreasing, offsets[count] <= its length), each searched as if it were the
 * whole sequence -- window clipping at 0 and at the segment's own length, positions in the results segment-local.
 * The limits are the already normalised ones of LevenshteinSearchParams (as for fzb_find_near_matches), and the route
 * follows choose_search_class and the rules of the single-sequence entry points: exact (max_l_dist == 0), Hamming,
 * Levenshtein n-grams / LP, generic n-grams / LP -- chosen from m and the limits only, never from a segment's length.
 * Segments of up to FZB_SEG_SHORT_BYTES are searched by one warp each (five kernel launches per call, whatever
 * `count`); a longer segment is copied device-to-device into a workspace and searched with the single-sequence entry
 * points (their launches add to stats.n_launches).  stats.route = 8 (segments).
 * Lists (fzb_result_copy) are segment-major; fzb_result_segment_counts gives each segment's share:
 *   FZB_FINAL  each segment's consolidate_matches result in (start, end, dist) order (exact / Hamming: its raw list);
 *   FZB_RAW    each segment's raw multiset in (start, end, dist) order -- NOT the reference's generation order;
 *              no anchors.
 * FZB_F_GLOBAL and sharded handles are refused (FZB_E_INVALID); more than FZB_SEG_MAX_COUNT segments per call
 * (the segment number travels in 23 bits of each raw record) is FZB_E_UNSUPPORTED.
 */
#define FZB_SEG_SHORT_BYTES 4096
#define FZB_SEG_MAX_COUNT (1u << 23)
int fzb_search_segments(fzb_haystack *h, const uint8_t *pattern, uint32_t m, const uint64_t *offsets, uint64_t count,
                        uint32_t max_subs, uint32_t max_ins, uint32_t max_dels, uint32_t max_l_dist, uint32_t flags,
                        fzb_result **out);
/* counts[0 .. count) = the length of each segment's `which` list (results of fzb_search_segments only). */
int fzb_result_segment_counts(const fzb_result *r, int which, uint64_t *counts);

/* ExactSearch.search (search_exact.py:80-85): all (overlapping) occurrences. FINAL == RAW. */
int fzb_search_exact(fzb_haystack *h, const uint8_t *pattern, uint32_t m, uint32_t flags,
                     fzb_result **out);
/* search_exact(subsequence, sequence, start_index, end_index) (search_exact.py:22-56; _common.c:5-112): the
 * occurrences lying wholly inside [start, end), both clamped as the reference clamps them (:29-30).  Only
 * the window is scanned.  Whole-sequence handles only. */
int fzb_search_exact_window(fzb_haystack *h, const uint8_t *pattern, uint32_t m, uint64_t start, uint64_t end,
                            uint32_t flags, fzb_result **out);

/*
 * One-shot convenience with HOST buffers (what find_near_matches() does): upload, dispatch like
 * choose_search_class (__init__.py:60-83) on the already normalised limits, search, consolidate.
 */
int fzb_find_near_matches(const uint8_t *pattern, uint32_t m, const uint8_t *haystack, uint64_t n,
                          uint32_t max_subs, uint32_t max_ins, uint32_t max_dels,
                          uint32_t max_l_dist, int device, fzb_result **out);

/*
 * "Is there any near-match?" -- the boolean form of the four searches (has_near_match_substitutions_lp /
 * _ngrams, substitutions_only.py:18-34,139-145,218-233; has_near_match_generic_ngrams, generic_search.py:240-253;
 * substitutions_only_has_near_matches_*_byteslike, _substitutions_only.c:4-17), with early termination: the
 * resident sequence is searched in chunks of growing size and the call returns after the first chunk that holds
 * a match.  Limits are the already normalised ones of LevenshteinSearchParams (as for fzb_find_near_matches).
 * *found = 1 iff find_near_matches would return a non-empty list.
 */
int fzb_has_near_match(fzb_haystack *h, const uint8_t *pattern, uint32_t m, uint32_t max_subs,
                       uint32_t max_ins, uint32_t max_dels, uint32_t max_l_dist, int *found);

/* fzb_find_near_matches keeps one device workspace per device (haystack buffer, bitmap, staging)
 * alive between calls so that a call costs one H2D copy + the kernels; this frees them. */
void fzb_release_workspace(void);

uint64_t fzb_result_count(const fzb_result *r, int which);
/* Copy out `which` list; any pointer may be NULL.  anchor_ngram / anchor_idx are only meaningful
 * for the RAW list of n-gram searches (n-gram ordinal and hit index), else -1. */
int fzb_result_copy(const fzb_result *r, int which, int64_t *start, int64_t *end, int32_t *dist,
                    int32_t *anchor_ngram, int64_t *anchor_idx);

/* For the FINAL list: the hull [hull_start, hull_end) of the group of overlapping raw matches each
 * final match won (for the unconsolidated routes: the match itself). */
int fzb_result_hulls(const fzb_result *r, int64_t *hull_start, int64_t *hull_end);

/* FINAL list as rows (start, end, dist, hull_start, hull_end), at most max_rows of them, straight
 * into a caller buffer (e.g. the pinned send buffer of the multi-GPU all-gather).  Returns the total
 * number of groups (which may exceed max_rows) or a negative error. */
int64_t fzb_result_group_rows(const fzb_result *r, int64_t *rows, uint64_t max_rows);

typedef struct fzb_stats_s {
    double gpu_ms;          /* CUDA-event time of all kernels of the search */
    double filter_ms;       /* ... of the haystack scan (filter) kernel alone */
    uint64_t bytes_scanned; /* haystack bytes the scan kernel read (algorithmic bytes) */
    uint64_t n_candidates;  /* granules / windows handed to the verify stage */
    uint32_t n_launches;    /* kernels launched */
    uint32_t route;         /* 0 exact, 1 n-grams (sampled filter), 2 n-grams (dense filter), 3 LP,
                               4 hamming, 5 generic n-grams, 6 generic LP, 8 segments (fzb_search_segments) */
} fzb_stats;
int fzb_result_stats(const fzb_result *r, fzb_stats *out);
void fzb_result_destroy(fzb_result *r);

/* consolidate_overlapping_matches (common.py:185-189) on caller-supplied triples (used to merge
 * per-shard raw streams after the multi-GPU gather).  Writes at most n winners; returns the count
 * (>= 0) or a negative error. */
int64_t fzb_consolidate(const int64_t *start, const int64_t *end, const int32_t *dist, uint64_t n,
                        int64_t *out_start, int64_t *out_end, int32_t *out_dist);

/* Like fzb_consolidate but writes one row (start, end, dist, hull_start, hull_end) per group into
 * out_rows[n][5] -- the per-shard input of fzb_merge_groups. Returns the number of groups. */
int64_t fzb_consolidate_groups(const int64_t *start, const int64_t *end, const int32_t *dist, uint64_t n,
                               int64_t *out_rows);

/* Multi-GPU merge: rows[n][5] = (start, end, dist, hull_start, hull_end), one row per group found by
 * any shard (fzb_result_copy(FINAL) + fzb_result_hulls of every shard, concatenated).  Writes the
 * global consolidated list (at most n rows); returns its length or a negative error. */
int64_t fzb_merge_groups(const int64_t *rows, uint64_t n, int64_t *out_start, int64_t *out_end,
                         int32_t *out_dist);

/*
 * TEST HOOK (not part of the search API): runs the expansion routines of the verify kernels -- the device
 * restatement of _expand / _py_expand_short / _py_expand_long (levenshtein_ngram.py:8-143; the Cython
 * seams c_expand_short / c_expand_long, _levenshtein_ngrams.pyx:9-154, are what a per-candidate FFI would
 * bind) -- on `count` caller-supplied cases: case i is (subs[sub_off[i]:sub_off[i+1]],
 * seqs[seq_off[i]:seq_off[i+1]], max_l[i]); variant[i] = 0 (_expand's own choice), 1 (short), 2 (long).
 * out[8*i..8*i+7] = (dist, len) from four device code paths: bit-parallel forwards / backwards (the right- and
 * left-expansion forms), cell-by-cell forwards / backwards; (-1,-1) = (None, None), (-2,-2) = path not applicable.
 */
int fzb_debug_expand(const uint8_t *subs, const uint32_t *sub_off, const uint8_t *seqs,
                     const uint32_t *seq_off, const int32_t *max_l, const int32_t *variant, uint32_t count,
                     int device, int32_t *out);

/* TEST / PROFILING HOOK: out[0..15] = the 16 device counters of the handle's last search (candidates, raw
 * records, final groups, and in slots 10-13 the phase times of k_post's last CTA in nanoseconds); out[16..31] =
 * the header of its last multi-GPU merge (status, global count, epoch, -, ns waiting for peers, ns merging,
 * non-head rows). */
int fzb_debug_counters(const fzb_haystack *h, uint32_t out[32]);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* FUZZB200_H */
