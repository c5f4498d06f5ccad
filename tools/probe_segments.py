#!/usr/bin/env python
"""One pattern over many sequences: find_near_matches_in_sequences (fzb_search_segments) vs the per-item loop.

Prints one JSON line per workload (all seeded; mutated copies of the primer planted at segment starts, middles and
ends):
  reads-lev    10^6 DNA reads of 150 bytes, primer of 20, max_l_dist=2
  reads-ham    the same reads, max_substitutions=2 (no insertions / deletions)
  lines-lev    10^5 ASCII lines of 1 KiB, max_l_dist=2
  long-lev     64 sequences of 1 MiB, max_l_dist=2 (above the short-segment bound: one single-sequence search each)
  mix-lev      a mix of the above (2*10^5 reads, 2*10^4 lines, 8 long sequences), max_l_dist=2
and, with --bound, reads of 2, 3, 4, 5 and 8 KiB searched both ways (warp kernels / single-sequence search), which is
the measurement behind FZB_SEG_SHORT_BYTES.

Per workload: device time of the segmented call (CUDA events on the handle's stream around it), end-to-end time of
find_near_matches_in_sequences with the Match objects built, the per-item find_near_matches loop through this
library on the first 10 000 items (a SAMPLE, reported as a per-item rate), the reference (oracle/_ref) over all host
cores on a sample (core count stated), and a parity check against oracle.find_near_matches (every segment of the
two smallest workloads, a seeded sample of the others).  The GPU's name and power limit come from a read-only
nvidia-smi query in the same run.  Usage: python tools/probe_segments.py [--bound] [--quick]
"""
import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import oracle  # noqa: E402
from fuzzysearch_b200 import _native, find_near_matches, find_near_matches_in_sequences  # noqa: E402
from fuzzysearch_b200 import search as _search  # noqa: E402

DNA, ASCII = b"ACGT", bytes(range(32, 127))
BIG = 1 << 29


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception as e:  # noqa: BLE001
        return "unknown (%r)" % e, "unknown"


def make_items(seed, count, length, alphabet, primer):
    rng = np.random.default_rng(seed)
    alpha = np.frombuffer(alphabet, dtype=np.uint8)
    buf = alpha[rng.integers(0, len(alpha), size=count * length, dtype=np.int64)].reshape(count, length)
    m = len(primer)
    p = np.frombuffer(primer, dtype=np.uint8)
    for where, frac in ((0, 0.1), (1, 0.1), (2, 0.1)):
        rows = np.nonzero(rng.random(count) < frac)[0]
        pos = {0: 0, 1: (length - m) // 2, 2: length - m}[where]
        v = np.repeat(p[None, :], len(rows), axis=0)
        e = rng.integers(0, m, size=(len(rows), 2))  # up to two substitutions
        v[np.arange(len(rows)), e[:, 0]] = alpha[rng.integers(0, len(alpha), size=len(rows))]
        v[np.arange(len(rows)), e[:, 1]] = alpha[rng.integers(0, len(alpha), size=len(rows))]
        buf[rows, pos:pos + m] = v
    return [bytes(r) for r in buf]


def _ref_worker(args):
    items, primer, kw = args
    sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))
    import fuzzysearch as fz
    t = time.perf_counter()
    for s in items:
        fz.find_near_matches(primer, s, **kw)
    return time.perf_counter() - t


def reference_rate(items, primer, kw, cores, budget_items):
    """items per second of the reference over `cores` processes, on the first budget_items items."""
    if not os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "fuzzysearch")):
        return None
    sample = items[:budget_items]
    chunks = [sample[i::cores] for i in range(cores)]
    with mp.get_context("fork").Pool(cores) as pool:
        pool.map(_ref_worker, [(c[:2], primer, kw) for c in chunks])  # import + warm
        t = time.perf_counter()
        pool.map(_ref_worker, [(c, primer, kw) for c in chunks])
        dt = time.perf_counter() - t
    return len(sample) / dt


def device_time(items, primer, kw):
    """CUDA-event time of the segmented call alone (the items already resident)."""
    subs, ins, dels, l = oracle.normalize_params(kw.get("max_substitutions"), kw.get("max_insertions"),
                                                 kw.get("max_deletions"), kw.get("max_l_dist"))
    lim = [BIG if x is None else min(x, BIG) for x in (subs, ins, dels)] + [l]
    blob = b"".join(items)
    offsets = np.zeros(len(items) + 1, dtype=np.uint64)
    np.cumsum([len(s) for s in items], out=offsets[1:])
    hay = _native.Haystack.from_host(blob)
    res = hay.search_segments(primer, offsets, *lim)  # warm-up
    res.close()
    hay.timer_start()
    res = hay.search_segments(primer, offsets, *lim)
    ms = hay.timer_stop()
    st = res.stats()
    res.close()
    hay.close()
    return ms, st


def parity(items, got, primer, kw, idx):
    bad = 0
    for i in idx:
        exp = oracle.find_near_matches(primer, items[i], **kw)
        ours = [(x.start, x.end, x.dist) for x in got[i]]
        if ours != exp:
            # ties inside a group may legitimately differ only where the oracle's winner is not unique
            fin, raw = oracle.find_near_matches(primer, items[i], return_raw=True, **kw)
            from parity import is_admissible_final
            if not is_admissible_final(ours, raw):
                bad += 1
    return bad


def run(name, items, primer, kw, full_parity, args, gpu):
    n_bytes = sum(len(s) for s in items)
    dev_ms, st = device_time(items, primer, kw)
    find_near_matches_in_sequences(primer, items[:100], **kw)  # warm the workspace
    t = time.perf_counter()
    got = find_near_matches_in_sequences(primer, items, **kw)
    e2e = time.perf_counter() - t
    n_loop = min(len(items), 10000 if not args.quick else 500)
    t = time.perf_counter()
    for s in items[:n_loop]:
        find_near_matches(primer, s, **kw)
    loop_rate = n_loop / (time.perf_counter() - t)
    cores = os.cpu_count()
    ref_rate = reference_rate(items, primer, kw, cores, min(len(items), 200 * cores if not args.quick else 50))
    rng = np.random.default_rng(11)
    idx = range(len(items)) if full_parity else rng.choice(len(items), size=min(len(items), 20000), replace=False)
    bad = parity(items, got, primer, kw, idx)
    line = {"workload": name, "items": len(items), "bytes": n_bytes, "limits": kw,
            "device_ms": round(dev_ms, 3), "n_launches": st["n_launches"],
            "end_to_end_s": round(e2e, 4), "end_to_end_items_per_s": round(len(items) / e2e, 1),
            "matches": sum(len(g) for g in got),
            "per_item_loop_sample": {"items": n_loop, "items_per_s": round(loop_rate, 1),
                                     "projected_s": round(len(items) / loop_rate, 2)},
            "speedup_vs_per_item_loop": round(len(items) / loop_rate / e2e, 2),
            "reference_cpu": None if ref_rate is None else {"cores": cores, "items_per_s": round(ref_rate, 1),
                                                            "projected_s": round(len(items) / ref_rate, 2)},
            "parity": {"checked": len(idx), "mismatches": bad, "ok": bad == 0,
                       "scope": "every segment" if full_parity else "seeded sample"},
            "gpu": gpu[0], "power_limit": gpu[1]}
    print(json.dumps(line), flush=True)
    return bad == 0


def bound_sweep(gpu):
    """Reads of growing length searched by the warp kernels and, for comparison, by one single-sequence search each
    (what a segment above the bound gets): device time per read."""
    primer = make_items(5, 1, 20, DNA, b"A" * 20)[0]
    for length in (1024, 2048, 3072, 4096, 5120, 8192):
        count = max(64, (32 << 20) // length)
        items = make_items(length, count, length, DNA, primer)
        ms, _ = device_time(items, primer, dict(max_l_dist=2))
        hay = _native.Haystack.from_host(items[0])
        one = []
        for s in items[:64]:
            hay.upload(s)
            hay.timer_start()
            r = hay.search_levenshtein(primer, 2)
            one.append(hay.timer_stop())
            r.close()
        hay.close()
        print(json.dumps({"bound_sweep": True, "read_bytes": length, "reads": count,
                          "warp_kernels_us_per_read": round(1000 * ms / count, 3),
                          "single_search_us_per_read": round(1000 * float(np.median(one[4:])), 3),
                          "gpu": gpu[0], "power_limit": gpu[1]}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true", help="tiny sizes (a rehearsal of the script, no numbers)")
    ap.add_argument("--bound", action="store_true", help="also the sweep behind FZB_SEG_SHORT_BYTES")
    args = ap.parse_args()
    gpu = gpu_info()
    scale = 1000 if args.quick else 1
    primer = make_items(1, 1, 20, DNA, b"A" * 20)[0]
    reads = make_items(2, 10 ** 6 // scale, 150, DNA, primer)
    lprimer = make_items(3, 1, 20, ASCII, b"A" * 20)[0]
    lines = make_items(4, 10 ** 5 // scale, 1024, ASCII, lprimer)
    longs = make_items(6, 64 if not args.quick else 2, (1 << 20) // scale, DNA, primer)
    ok = True
    ok &= run("reads-lev", reads, primer, dict(max_l_dist=2), False, args, gpu)
    ok &= run("reads-ham", reads, primer, dict(max_substitutions=2, max_insertions=0, max_deletions=0), False,
              args, gpu)
    ok &= run("lines-lev", lines, lprimer, dict(max_l_dist=2), True, args, gpu)
    ok &= run("long-lev", longs, primer, dict(max_l_dist=2), True, args, gpu)
    mix = reads[:len(reads) // 5] + lines[:len(lines) // 5] + longs[:8]
    np.random.default_rng(9).shuffle(mix)
    ok &= run("mix-lev", mix, primer, dict(max_l_dist=2), False, args, gpu)
    if args.bound:
        bound_sweep(gpu)
    _search.release_workspace()
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
