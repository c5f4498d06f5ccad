#!/usr/bin/env python
"""bench.py -- the driver's benchmark contract for the fuzzysearch hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload ...] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input: ONE bounded-Levenshtein
search (``find_near_matches(pattern, haystack, max_l_dist=2)``, |pattern| = 20) of a 4 GiB
95-symbol ASCII haystack per GPU (BASELINE.json configs[1]; with N GPUs the global sequence is
N x 4 GiB, sharded with a halo of |pattern|+k = configs[3], weak scaling).

* ``value``  = haystack GB/s scanned, whole job, inputs resident in HBM, timed on the device (CUDA
  events on the library's stream around exactly K searches incl. result read-back; max over ranks).
* ``e2e``    = same metric through the C-ABI one-shot call with HOST (pinned) buffers: H2D copy of
  the haystack and D2H of the matches inside the timed region.
* ``roofline`` = the dominant kernel (k_filter_sampled): algorithmic bytes (1 per haystack byte) /
  its CUDA-event duration, against the measured HBM peak of MEASURED_PEAKS.json.
* ``cpu_baseline`` / ``--impl reference`` = the reference itself (oracle/_ref, compiled from
  /root/reference by oracle/build_ref.py) on the box's host cores, on a bounded sample.

Inputs are far larger than L2 (4 GiB vs 126 MB), so no explicit L2 flush is needed between steps.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ASCII = bytes(range(32, 127))
DNA = b"ACGT"
GiB = 1 << 30

WORKLOADS = {
    # name: (alphabet, bytes per GPU, m, search kind, k)
    "ascii4g_lev_m20_k2": (ASCII, 4 * GiB, 20, "lev", 2),
    "dna4g_ham_m32_k3": (DNA, 4 * GiB, 32, "ham", 3),
    "dna4g_lev_m20_k2": (DNA, 4 * GiB, 20, "lev", 2),       # configs[0]'s corpus at scale (dense filter route)
    "ascii64m_lev_m20_k2": (ASCII, 64 << 20, 20, "lev", 2),  # quick self-test size
    # BASELINE.json configs[4]: 1024 patterns |p| in [8,64], k in [1,4] over one 4 GiB haystack; a step is
    # the whole batch (round 1: one pass per pattern); m and k below are only used for the halo
    "ascii4g_batch1024": (ASCII, 4 * GiB, 64, "batch", 4),
}


def mutate(rng, pat, alphabet, nedits, subs_only):
    s = bytearray(pat)
    for _ in range(nedits):
        op = 0 if subs_only else int(rng.integers(3))
        if op == 0:
            s[int(rng.integers(len(s)))] = alphabet[int(rng.integers(len(alphabet)))]
        elif op == 1:
            s.insert(int(rng.integers(len(s) + 1)), alphabet[int(rng.integers(len(alphabet)))])
        else:
            del s[int(rng.integers(len(s)))]
    return bytes(s)


def make_plants(seed, lo, hi, m, k, pat, alphabet, n_plants, subs_only):
    """Deterministic plants inside [lo, hi): (global offset, bytes).  0..k+1 edits each (k+1 are
    negatives), plus overlapping clusters for the consolidation."""
    rng = np.random.default_rng(seed)
    out = []
    span = (hi - lo - 8 * m) // n_plants
    for i in range(n_plants):
        pos = lo + 4 * m + i * span + int(rng.integers(0, span - 4 * m))
        out.append((pos, mutate(rng, pat, alphabet, int(rng.integers(0, k + 2)), subs_only)))
    for c in range(16):
        pos = lo + 4 * m + int(rng.integers(0, hi - lo - 16 * m))
        out.append((pos, pat + pat[m // 2:] + pat))
    return out


def clocks_monitor_start(path, gpu_index):
    try:
        return subprocess.Popen(
            ["nvidia-smi", "-i", str(gpu_index),
             "--query-gpu=index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap",
             "--format=csv,noheader,nounits", "-lms", "100"],
            stdout=open(path, "w"), stderr=subprocess.DEVNULL)
    except OSError:
        return None


def clocks_monitor_stop(proc, path):
    if proc is None:
        return None
    proc.terminate()
    try:
        proc.wait(timeout=5)
    except subprocess.TimeoutExpired:
        proc.kill()
    sm, mx, reasons = [], [], set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    try:
        for line in open(path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
    except OSError:
        return None
    if not sm:
        return None
    # "under load": the upper half of the samples (the monitor also sees the idle edges)
    load = sorted(sm)[len(sm) // 2:]
    return {"sm_mhz": float(np.median(load)), "sm_max_mhz": float(max(mx)), "samples": len(sm),
            "reasons": sorted(reasons)}


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        v = json.load(open(p))
        return float(v["hbm_gbs"]), "measured (MEASURED_PEAKS.json, copy read+write)"
    except (OSError, KeyError, ValueError):
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture, or None."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "filter_traffic.json")))
    except (OSError, ValueError):
        return None


# -------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation (oracle/_ref), all host cores
# -------------------------------------------------------------------------------------------------
_REF_STATE = {}


def _ref_worker(args):
    lo, hi, kind, k = args
    fz = _REF_STATE["fz"]
    pat = _REF_STATE["pat"]
    chunk = _REF_STATE["hay"][lo:hi].tobytes()
    if kind == "lev":
        ms = fz.find_near_matches(pat, chunk, max_l_dist=k)
    else:
        ms = fz.find_near_matches(pat, chunk, max_substitutions=k, max_insertions=0, max_deletions=0)
    return [(m.start + lo, m.end + lo, m.dist) for m in ms]


def reference_available():
    return os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "fuzzysearch"))


def import_reference():
    sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))
    import fuzzysearch
    return fuzzysearch


def run_reference_sample(hay, pat, kind, k, cores, repeats=1):
    """Time the reference on `hay` (numpy uint8) split into overlapping chunks over `cores`
    processes (the reference's own chunk + carry-over rule, __init__.py:135-138).  Returns
    (seconds, n_matches).  With cores == 1 it is one plain find_near_matches call."""
    import multiprocessing as mp
    fz = import_reference()
    _REF_STATE.update(fz=fz, pat=pat, hay=hay)
    n = hay.size
    m = len(pat)
    keep = m - 1 + (k if kind == "lev" else 0)
    best = None
    nm = 0
    if cores == 1:
        for _ in range(repeats):
            t0 = time.perf_counter()
            res = _ref_worker((0, n, kind, k))
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
            nm = len(res)
        return best, nm
    nchunks = cores * 4
    step = (n + nchunks - 1) // nchunks
    tasks = [(max(0, i * step), min(n, (i + 1) * step + keep), kind, k) for i in range(nchunks)
             if i * step < n]
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        pool.map(_ref_worker, tasks[:cores])  # warm the workers
        for _ in range(repeats):
            t0 = time.perf_counter()
            parts = pool.map(_ref_worker, tasks, chunksize=1)
            allm = [x for p in parts for x in p]
            if kind == "lev" and allm:
                # one global consolidation of the per-chunk winners (find_near_matches_in_file,
                # __init__.py:126), with the reference's own function
                Match = fz.Match
                from fuzzysearch.common import consolidate_overlapping_matches
                allm = consolidate_overlapping_matches([Match(s, e, d, b"") for s, e, d in allm])
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
            nm = len(allm)
    return best, nm


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def synth_sample_host(alphabet, seed, pat, nbytes, m, k, kind):
    """The first `nbytes` of rank 0's corpus, regenerated on the host (counter-based generator +
    the same plants), so the CPU baseline scans the same bytes the GPU scans.  Uses the oracle's
    restatement of the generator (oracle/fzoracle.c: fzo_synth): the reference arm never loads the
    product library."""
    import oracle
    hay = oracle.synth(0, nbytes, alphabet, seed)
    for pos, b in make_plants(seed + 1, 0, nbytes, m, k, pat, alphabet, max(8, nbytes >> 20), kind == "ham"):
        b = b[:max(0, nbytes - pos)]
        hay[pos:pos + len(b)] = np.frombuffer(b, dtype=np.uint8)
    return hay


# -------------------------------------------------------------------------------------------------
# parity inside the numbers: the C oracle over this rank's WHOLE shard, compared with the device
# -------------------------------------------------------------------------------------------------
def parity_check(F, hs, pat, kind, k, blo, bhi, own_lo, own_hi, global_final, dist, rank, world):
    """Runs the CPU oracle (oracle/fzoracle.c, the pinned restatement of the reference's pure-Python
    path) over every byte of this rank's shard buffer and compares
      * the device's raw match stream of the shard, element for element in generation order, with the
        oracle's stream restricted to the anchors this rank owns (owned anchors see exactly the same
        window in the shard buffer as in the global sequence: the halo is len(pattern)+k);
      * the (global) final list with consolidate_overlapping_matches over all ranks' oracle streams.
    -> the "parity" object of the JSON line (rank 0; other ranks return None)."""
    import oracle
    t0 = time.perf_counter()
    host = np.empty(bhi - blo, dtype=np.uint8)
    chunk = 256 << 20
    for off in range(0, bhi - blo, chunk):
        nb = min(chunk, bhi - blo - off)
        host[off:off + nb] = np.frombuffer(hs.read(blo + off, nb), dtype=np.uint8)
    t1 = time.perf_counter()
    if kind == "lev":
        raw_o, ng_o, ix_o = oracle.levenshtein_ngrams_raw(pat, host, k, with_anchor=True)
        raw_o = raw_o.copy()
        raw_o[:, 0:2] += blo
        ix_o = ix_o + blo
        keep = (ix_o >= own_lo) & (ix_o < own_hi)
        raw_o, ng_o, ix_o = raw_o[keep], ng_o[keep], ix_o[keep]
        res = hs.search_levenshtein(pat, k, F.F_NO_FINAL)
        s, e, d, ng, ix = res.arrays(F.RAW, anchors=True)
        res.close()
        raw_ok = (len(s) == len(raw_o) and bool(np.array_equal(s, raw_o[:, 0])) and
                  bool(np.array_equal(e, raw_o[:, 1])) and bool(np.array_equal(d, raw_o[:, 2])) and
                  bool(np.array_equal(ng, ng_o)) and bool(np.array_equal(ix, ix_o)))
    else:
        raw_o = oracle.substitutions(pat, host, k).copy()
        raw_o[:, 0:2] += blo
        keep = (raw_o[:, 0] >= own_lo) & (raw_o[:, 0] < own_hi)
        raw_o = raw_o[keep]
        res = hs.search_hamming(pat, k)
        s, e, d = res.arrays(F.RAW)
        res.close()
        raw_ok = (len(s) == len(raw_o) and bool(np.array_equal(s, raw_o[:, 0])) and
                  bool(np.array_equal(e, raw_o[:, 1])) and bool(np.array_equal(d, raw_o[:, 2])))
    t2 = time.perf_counter()
    n_raw_dev = len(s)
    parts, oks, nraw, nbytes = [raw_o], [raw_ok], [n_raw_dev], [bhi - blo]
    if dist is not None:
        box = [None] * world
        dist.all_gather_object(box, (raw_o, raw_ok, n_raw_dev, bhi - blo))
        parts, oks, nraw, nbytes = [b[0] for b in box], [b[1] for b in box], [b[2] for b in box], [b[3] for b in box]
    if rank != 0:
        return None
    all_raw = np.concatenate(parts, axis=0) if parts else np.zeros((0, 3), np.int64)
    if kind == "lev":
        want = [tuple(int(x) for x in r) for r in oracle.consolidate(all_raw)]
    else:
        want = sorted(tuple(int(x) for x in r) for r in all_raw)
    final_ok = list(global_final) == want
    return {"oracle": "oracle/fzoracle.c over every byte of every rank's shard (+halo)",
            "checked_bytes": int(sum(nbytes)), "raw": int(sum(nraw)), "raw_ok": bool(all(oks)),
            "final": len(want), "final_ok": bool(final_ok), "ok": bool(all(oks) and final_ok),
            "d2h_s": round(t1 - t0, 2), "oracle_s": round(t2 - t1, 2)}


def batch_parity(F, hs, pats, ks, n):
    """Parity of the 1024-pattern batch at full size (untimed): (1) EVERY pattern's final list from the batch call
    equals the single-pattern search of the same 4 GiB (the path whose whole-shard oracle comparison is the
    headline's "parity" block); (2) the CPU oracle directly, for a sample of patterns of every route: over a window
    around each match the batch reported (same matches, nothing else nearby) and over a 16 MiB prefix of the
    sequence (nothing missed, nothing invented in the bulk)."""
    import oracle
    results, _ = hs.search_levenshtein_batch(pats, ks)
    finals, route_of = [], []
    for r in results:
        finals.append(r.triples(F.FINAL))
        route_of.append(r.stats()["route"])
        r.close()
    differ = []
    for i, (bp, bk) in enumerate(zip(pats, ks)):
        r = hs.search_levenshtein(bp, bk)
        if r.triples(F.FINAL) != finals[i]:
            differ.append(i)
        r.close()
    sample, seen = [], {}
    for i, rt in enumerate(route_of):  # the first 8 patterns of every route
        if seen.setdefault(rt, 0) < 8:
            seen[rt] += 1
            sample.append(i)
    margin, pad = 512, 4096
    win_ok, n_windows = True, 0
    for i in sample:
        bp, bk = pats[i], ks[i]
        for s0, e0, _ in finals[i]:
            lo, hi = max(0, s0 - pad), min(n, e0 + pad)
            host = hs.read(lo, hi - lo)
            inner = lambda t: (t[0] >= lo + margin or lo == 0) and (t[1] <= hi - margin or hi == n)  # noqa: E731
            want = [(a + lo, b + lo, d) for a, b, d in oracle.find_near_matches(bp, host, max_l_dist=bk)]
            got = [t for t in finals[i] if t[0] >= lo and t[1] <= hi]
            win_ok &= [t for t in want if inner(t)] == [t for t in got if inner(t)]
            n_windows += 1
    plen = 16 << 20
    prefix = hs.read(0, plen)
    pre_ok = True
    pre_ids = sample[::4][:6]
    for i in pre_ids:
        want = [t for t in oracle.find_near_matches(pats[i], prefix, max_l_dist=ks[i]) if t[1] <= plen - margin]
        pre_ok &= want == [t for t in finals[i] if t[1] <= plen - margin]
    return {"patterns_vs_single_search": len(pats), "differing": differ[:8], "single_ok": not differ,
            "oracle_windows": n_windows, "oracle_windows_ok": bool(win_ok),
            "oracle_prefix_bytes": plen, "oracle_prefix_patterns": len(pre_ids), "oracle_prefix_ok": bool(pre_ok),
            "ok": bool(not differ and win_ok and pre_ok)}


# -------------------------------------------------------------------------------------------------
# secondary workloads: short, driver-visible runs of the other BASELINE configs on one GPU
# -------------------------------------------------------------------------------------------------
def run_secondary(F, main_hs, main_alphabet, seed, peak):
    """-> {name: {...}}: configs[2] (4 GiB DNA, substitutions only), configs[0]'s corpus at 4 GiB (DNA Levenshtein,
    dense-filter route) and configs[4] (1024-pattern batch over the resident ASCII haystack).  Device-resident
    inputs, CUDA events on the library's stream; same 4 GiB size as the headline."""
    out = {}
    n = 4 * GiB

    def timed(hs, fn, steps, warm):
        for _ in range(warm):
            fn()
        filt, cnt = [], 0
        hs.timer_start()
        for _ in range(steps):
            st, cnt = fn()
            filt.append(st["filter_ms"])
        ms = hs.timer_stop() / steps
        return ms, float(np.mean(filt)), cnt

    try:
        dna = F.Haystack.alloc(n)
        dna.fill_synthetic(DNA, seed + 7)
        rng = np.random.default_rng(seed + 7)
        a = np.frombuffer(DNA, dtype=np.uint8)
        for name, m, k, kind in (("dna4g_ham_m32_k3", 32, 3, "ham"), ("dna4g_lev_m20_k2", 20, 2, "lev")):
            pat = bytes(a[rng.integers(0, 4, size=m)])
            for pos, b in make_plants(seed + 8 + m, 0, n, m, k, pat, DNA, 4096, kind == "ham"):
                dna.write(pos, b)

            def one(pat=pat, k=k, kind=kind):
                r = dna.search_hamming(pat, k) if kind == "ham" else dna.search_levenshtein(pat, k)
                st, c = r.stats(), r.count(F.FINAL)
                r.close()
                return st, c
            ms, filt, cnt = timed(dna, one, 10, 3)
            out[name] = {"value": n / (ms * 1e-3) / 1e9, "unit": "GB/s", "ms_per_step": ms, "steps": 10, "warmup": 3,
                         "matches_per_step": int(cnt),
                         "roofline": {"kernel": "k_hamming_count" if kind == "ham" else "k_filter_dense",
                                      "kernel_ms": filt, "achieved": n / (filt * 1e-3) / 1e9, "peak": peak,
                                      "frac": n / (filt * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": n}}
        dna.close()
    except Exception as e:  # noqa: BLE001 -- the headline line must still be printed
        out["dna_error"] = repr(e)[:200]
    try:
        brng = np.random.default_rng(seed + 99)
        alpha = np.frombuffer(main_alphabet, dtype=np.uint8)
        pats, ks = [], []
        for i in range(1024):
            bm, bk = int(brng.integers(8, 65)), int(brng.integers(1, 5))
            bp = bytes(alpha[brng.integers(0, len(alpha), size=bm)])
            pats.append(bp)
            ks.append(bk)
            for _ in range(8):
                pos = 1000 + int(brng.integers(0, n - 2000))
                main_hs.write(pos, mutate(brng, bp, main_alphabet, int(brng.integers(0, bk + 2)), False))
        routes = {}

        def batch():
            results, st = main_hs.search_levenshtein_batch(pats, ks)
            c = 0
            routes.clear()
            for r in results:
                c += r.count(F.FINAL)
                rs = r.stats()
                agg = routes.setdefault(rs["route"], [0, 0.0])
                agg[0] += 1
                agg[1] += rs["gpu_ms"]
                r.close()
            return st, c
        ms, _, cnt = timed(main_hs, batch, 2, 1)
        shared_ms = routes.get("ngrams/sampled-filter", [0, 0.0])[1]
        try:
            bparity = batch_parity(F, main_hs, pats, ks, n)
        except Exception as e:  # noqa: BLE001
            bparity = {"ok": False, "error": repr(e)[:200]}
        out["ascii4g_batch1024"] = {
            "value": n / (ms * 1e-3) / 1e9, "unit": "GB/s of haystack per 1024-pattern batch", "ms_per_step": ms,
            "steps": 2, "warmup": 1, "patterns": 1024, "pattern_GB_per_s": 1024 * n / (ms * 1e-3) / 1e9,
            "matches_per_step": int(cnt),
            "routes": {r: {"patterns": v[0], "device_ms": v[1]} for r, v in sorted(routes.items())},
            "parity": bparity,
            "roofline": {"kernel": "k_filter_multi + k_verify_multi (one scan for all lemma-eligible patterns)",
                         "kernel_ms": shared_ms, "achieved": n / (shared_ms * 1e-3) / 1e9 if shared_ms else 0.0,
                         "peak": peak, "frac": (n / (shared_ms * 1e-3) / 1e9 / peak) if shared_ms else 0.0,
                         "algorithmic_bytes_per_launch": n,
                         "note": "the shared scan reads the haystack once for its patterns; dense-filter and LP "
                                 "patterns still cost one pass each (whole-batch value above)"}}
    except Exception as e:  # noqa: BLE001
        out["batch_error"] = repr(e)[:200]
    return out


# -------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="ascii4g_lev_m20_k2", choices=sorted(WORKLOADS))
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the full-shard oracle comparison")
    ap.add_argument("--no-secondary", action="store_true", help="skip the short runs of the other configs")
    ap.add_argument("--cpu-sample-mib", type=int, default=0, help="0 = auto (about 10-20 s of CPU work)")
    ap.add_argument("--reduce", default="p2p", choices=["p2p", "nccl", "torch"],
                    help="multi-GPU reduction: inside the library over NVLink peer memory (default; 'nccl' is an "
                         "alias), or through torch.distributed (tools/torch_reduce.py, comparison only)")
    ap.add_argument("--ref-cores", type=int, default=0, help="reference arm: processes to use (0 = all cores)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the matches the last timed step returned to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what --impl ours computed")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    alphabet, per_gpu, m, kind, k = WORKLOADS[args.workload]
    seed = 20260923
    metric = "haystack_GB_per_s_scanned"
    unit = "GB/s"
    config = {"workload": args.workload, "alphabet": len(alphabet), "pattern_len": m,
              "max_l_dist" if kind == "lev" else "max_substitutions": k,
              "bytes_per_gpu": per_gpu, "global_bytes": per_gpu * world,
              "sharding": "contiguous shards, halo=%d, no data-path collective" % (m + k),
              "l2": "inputs larger than L2 (no flush needed)"}

    rng = np.random.default_rng(seed)
    pat = bytes(np.frombuffer(alphabet, dtype=np.uint8)[rng.integers(0, len(alphabet), size=m)])

    # ---------------------------------------------------------------------------------------------
    if args.impl == "reference":
        if world > 1 and rank != 0:
            return 0
        cores = args.ref_cores or host_cores()
        sample = (args.cpu_sample_mib << 20) if args.cpu_sample_mib else min(per_gpu, 1 * GiB)
        if not reference_available():
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref not built"}))
            return 0
        hay = synth_sample_host(alphabet, seed, pat, sample, m, k, kind)
        times, nm = [], 0
        for i in range(args.warmup + args.steps):
            dt, nm = run_reference_sample(hay, pat, kind, k, cores)
            if i >= args.warmup:
                times.append(dt)
        sec = float(np.median(times))
        val = sample / sec / 1e9
        # the reference as it actually ships is single-threaded: one plain find_near_matches call
        one_sample = min(sample, 256 << 20)
        one_sec, _ = run_reference_sample(hay[:one_sample], pat, kind, k, 1)
        line = {"impl": "reference", "metric": metric, "value": val, "unit": unit, "n_gpus": args.gpus,
                "steps": len(times), "warmup": args.warmup, "ms_per_step": sec * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
                "data": "synthetic", "config": config,
                "cpu_baseline": {"value": val, "unit": unit, "cores": cores, "kind": "reference",
                                 "sample": "first %d MiB of rank 0's corpus per step, split over %d "
                                           "processes with the reference's chunk overlap; value = median of "
                                           "%d steps" % (sample >> 20, cores, len(times)),
                                 "step_values": [sample / t / 1e9 for t in times],
                                 "single_core_value": one_sample / one_sec / 1e9,
                                 "single_core_sample": "one find_near_matches call over the first %d MiB"
                                                       % (one_sample >> 20)},
                "e2e": {"value": val, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0, "matches": nm}
        print(json.dumps(line))
        return 0

    # ---------------------------------------------------------------------------------------------
    from fuzzysearch_b200 import _native as F
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from fuzzysearch_b200.sharding import init_shard_comm, shard_bounds
    if args.reduce == "torch":  # comparison arm only: the same reduction through torch.distributed
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        from torch_reduce import gather_and_merge_groups

    # the single-pattern workloads shard the haystack (weak scaling: N x 4 GiB, configs[3]); the batch (configs[4]:
    # "1024 patterns over ONE 4 GiB haystack, 8 x B200") keeps the whole haystack on every GPU and splits the PATTERNS
    # (strong scaling: nothing to merge, every pattern's list is complete on the rank that searched it)
    global_len = per_gpu * world if kind != "batch" else per_gpu
    halo = m + k
    blo, bhi, own_lo, own_hi = (shard_bounds(global_len, world, rank, halo) if kind != "batch"
                                else (0, per_gpu, 0, per_gpu))
    if kind == "batch":
        config["global_bytes"] = per_gpu
        config["sharding"] = "haystack replicated, patterns split %d ways (pattern i on rank i %% N)" % world
    # device-resident shard generated ON the device (counter-based corpus keyed by global offset)
    hs = F.Haystack.alloc(bhi - blo, device=local_rank, buf_lo=blo, global_len=global_len, own_lo=own_lo,
                          own_hi=own_hi)
    hs.fill_synthetic(alphabet, seed)
    plants = []
    if kind == "batch":  # replicated haystack: the same corpus whatever N is
        plants = make_plants(seed + 1, 0, per_gpu, m, k, pat, alphabet, 4096, False)
    for r in range(world if kind != "batch" else 0):  # every rank knows every plant (needed for seam plants + checking)
        lo_r, hi_r = shard_bounds(global_len, world, r, halo)[2:]
        plants += make_plants(seed + 1 + r, lo_r, hi_r, m, k, pat, alphabet, 4096, kind == "ham")
        if r > 0:  # straddle the seam (tests/test_find_near_matches_in_file.py:84-86 deltas)
            for j, delta in enumerate((-m, -m + 1, -4, -2, -1, 0, 1)):
                plants.append((lo_r + delta + 256 * (j - 3), pat))
    for pos, b in plants:
        if pos >= blo and pos + len(b) <= bhi:
            hs.write(pos, b)

    in_library = world > 1 and args.reduce in ("p2p", "nccl") and kind != "batch"
    if in_library:
        init_shard_comm(hs)
        config["reduction"] = ("in-library, NVLink peer memory (k_push + k_merge on the search stream)"
                               if hs.p2p_enabled() else "in-library, staged NCCL all-gather + host merge")
    elif world > 1:
        config["reduction"] = "torch.distributed (tools/torch_reduce.py)"
    gflag = F.F_GLOBAL if in_library else 0

    batch_pats, batch_ks = [], []
    if kind == "batch":
        brng = np.random.default_rng(seed + 99)
        alpha = np.frombuffer(alphabet, dtype=np.uint8)
        for i in range(1024):
            bm, bk = int(brng.integers(8, 65)), int(brng.integers(1, 5))
            bp = bytes(alpha[brng.integers(0, len(alpha), size=bm)])
            batch_pats.append(bp)
            batch_ks.append(bk)
            for _ in range(8):
                pos = own_lo + 1000 + int(brng.integers(0, own_hi - own_lo - 2000))
                hs.write(pos, mutate(brng, bp, alphabet, int(brng.integers(0, bk + 2)), False))
        batch_pats, batch_ks = batch_pats[rank::world], batch_ks[rank::world]  # my share of the patterns

    def one_search(h):
        if kind == "lev":
            return h.search_levenshtein(pat, k, gflag)
        return h.search_hamming(pat, k, gflag)

    def step(h=None, keep=None):
        # one search of this rank's shard (local consolidation on the device); multi-GPU: the per-shard
        # groups are all-gathered by NCCL inside the library, on the search's stream, and merged
        # (--reduce torch: the same reduction through torch.distributed, for comparison).
        # With a list as `keep`, the results are appended to it instead of being closed.
        if kind == "batch":
            results, st = (h or hs).search_levenshtein_batch(batch_pats, batch_ks)
            nfinal = sum(r.count(F.FINAL) for r in results)
            if keep is not None:
                keep.extend(results)
                return st, nfinal
            for r in results:
                r.close()
            return st, nfinal
        res = one_search(h or hs)
        st = res.stats()
        if world > 1 and not in_library:
            merged = gather_and_merge_groups(result=res, as_arrays=True)
            nfinal = len(merged[0])
        else:
            merged = None
            nfinal = res.count(F.FINAL)
        if keep is not None:
            keep.append(res if merged is None else merged)
            if merged is None:
                return st, nfinal
        res.close()
        return st, nfinal

    def dump_outputs(kept):
        """What the caller of the timed path receives, as float64 columns: every final match (start, end,
        dist), plus the pattern index for the batch; a fixed sample of rows if they exceed 64 MiB."""
        if kind == "batch":
            cols = {"pattern": [], "start": [], "end": [], "dist": []}
            for j, r in enumerate(kept):  # this rank's patterns are rank, rank + world, ...
                s, e, d = r.arrays(F.FINAL)
                cols["pattern"].append(np.full(len(s), rank + j * world))
                cols["start"].append(s)
                cols["end"].append(e)
                cols["dist"].append(d)
                r.close()
            cols = {name: np.concatenate(c) if c else np.zeros(0) for name, c in cols.items()}
            if dist is not None:
                box = [None] * world
                dist.all_gather_object(box, cols)
                order = np.argsort(np.concatenate([b["pattern"] for b in box]), kind="stable")
                cols = {name: np.concatenate([b[name] for b in box])[order] for name in cols}
        else:
            r = kept[0]
            s, e, d = r if isinstance(r, tuple) else r.arrays(F.FINAL)
            if not isinstance(r, tuple):
                r.close()
            cols = {"start": s, "end": e, "dist": d}
        if rank != 0:
            return
        n = len(cols["start"])
        max_rows = (64 << 20) // (8 * (len(cols) + 1))  # + the "row" column of a sample
        if n > max_rows:
            rows = np.sort(np.random.default_rng(0).choice(n, max_rows, replace=False))
            cols = {name: c[rows] for name, c in cols.items()}
            cols["row"] = rows
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, c in cols.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), np.asarray(c, dtype=np.float64))

    def sync_all():
        if dist is not None:
            dist.barrier()
            import torch
            torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    clock_path = os.path.join(tempfile.gettempdir(), "fzb_clocks_%d.csv" % rank)
    mon = clocks_monitor_start(clock_path, local_rank) if rank == 0 else None
    time.sleep(0.3)
    sync_all()
    filt_ms, launches, nfinal = [], 0, 0
    kept = [] if args.dump_outputs else None
    hs.timer_start()
    t0 = time.perf_counter()
    for i in range(args.steps):
        st, nfinal = step(keep=kept if i == args.steps - 1 else None)
        filt_ms.append(st["filter_ms"])
        launches += st["n_launches"]
    dev_ms = hs.timer_stop()
    wall_ms = (time.perf_counter() - t0) * 1e3
    if kept is not None:
        dump_outputs(kept)
    sync_all()
    # the timed region of a default run lasts ~20 ms, shorter than one nvidia-smi sampling period: keep
    # the SAME searches running (untimed, same count on every rank) so the clock monitor sees the load
    soak = 0 if kind == "batch" else max(0, 400 - args.steps)
    for _ in range(soak):
        step()
    sync_all()
    time.sleep(0.2)
    clocks = clocks_monitor_stop(mon, clock_path)
    if clocks is not None:
        clocks["note"] = "sampled every 100 ms over the timed region plus %d identical untimed searches" % soak
    ms_per_step = dev_ms / args.steps
    if dist is not None:
        import torch
        t = torch.tensor([ms_per_step], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_per_step = float(t.item())
    value = global_len / (ms_per_step * 1e-3) / 1e9
    if dist is not None and kind == "batch":  # matches of all ranks' patterns
        import torch
        t = torch.tensor([nfinal], dtype=torch.int64, device="cuda")
        dist.all_reduce(t)
        nfinal = int(t.item())

    # ---- parity: the oracle over every byte of every shard vs the lists the timed searches return ----
    parity = None
    if not args.no_parity and kind in ("lev", "ham"):
        res = one_search(hs)
        if world > 1 and not in_library:
            gs, ge, gd = gather_and_merge_groups(result=res, as_arrays=True)
            gfinal = list(zip(gs.tolist(), ge.tolist(), gd.tolist()))
        else:
            gfinal = res.triples(F.FINAL)
        res.close()
        parity = parity_check(F, hs, pat, kind, k, blo, bhi, own_lo, own_hi, gfinal, dist, rank, world)

    # ---- end to end through the one-shot C-ABI call with pinned HOST buffers -----------------------
    e2e = None
    if args.e2e_steps > 0 and kind != "batch":
        pinned = F.PinnedBuffer(bhi - blo)
        chunk = 256 << 20
        for off in range(0, bhi - blo, chunk):  # host copy of the shard (setup, untimed)
            nb = min(chunk, bhi - blo - off)
            pinned.array[off:off + nb] = np.frombuffer(hs.read(blo + off, nb), dtype=np.uint8)
        subs, ins, dels, l = (k, k, k, k) if kind == "lev" else (k, 0, 0, k)

        h2 = None
        if world > 1:  # persistent shard handle: a step re-uploads the shard from pinned host memory
            h2 = F.Haystack.alloc(bhi - blo, device=local_rank, buf_lo=blo, global_len=global_len, own_lo=own_lo,
                                  own_hi=own_hi)
            if in_library:
                init_shard_comm(h2)

        def e2e_step():
            if world == 1:
                r = F.find_near_matches_host(pat, pinned.array, subs, ins, dels, l, device=local_rank)
                cnt = r.count(F.FINAL)
                d2h = cnt * 20
                r.close()
                return cnt, d2h
            h2.upload(pinned.array)
            _, nf = step(h2)
            return nf, nf * 40

        e2e_step()
        sync_all()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            cnt_e2e, d2h_bytes = e2e_step()
        sync_all()
        e2e_ms = (time.perf_counter() - t0) * 1e3 / args.e2e_steps
        if dist is not None:
            import torch
            t = torch.tensor([e2e_ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_ms = float(t.item())
        e2e = {"value": global_len / (e2e_ms * 1e-3) / 1e9, "unit": unit, "ms_per_step": e2e_ms,
               "h2d_bytes_per_step": (bhi - blo) + m, "d2h_bytes_per_step": int(d2h_bytes),
               "steps": args.e2e_steps, "timer": "host clock around the C-ABI call (includes H2D/D2H)",
               "matches": int(cnt_e2e), "input": "pinned host buffer"}
        if world == 1:
            # the drop-in call itself: fuzzysearch_b200.find_near_matches(pattern, <pageable bytes-like>, ...) ->
            # list[Match]; the upload goes through the library's pinned ring (host threads + DMA overlapped)
            import fuzzysearch_b200
            pageable = bytearray(bhi - blo)
            np.frombuffer(pageable, dtype=np.uint8)[:] = pinned.array
            kw = {"max_l_dist": k} if kind == "lev" else {"max_substitutions": k, "max_insertions": 0, "max_deletions": 0}
            fuzzysearch_b200.find_near_matches(pat, pageable, **kw)  # warm-up (ring allocation, page faults)
            times = []
            for _ in range(max(2, args.e2e_steps)):
                t0 = time.perf_counter()
                ms_list = fuzzysearch_b200.find_near_matches(pat, pageable, **kw)
                times.append(time.perf_counter() - t0)
            e2e["python"] = {"value": (bhi - blo) / float(np.median(times)) / 1e9, "unit": unit,
                             "ms_per_step": float(np.median(times)) * 1e3, "matches": len(ms_list),
                             "call": "fuzzysearch_b200.find_near_matches(pattern, bytearray (pageable), ...) -> list[Match]",
                             "h2d_bytes_per_step": bhi - blo}
            del pageable
        pinned.close()

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    peak, peak_src = hbm_peak()
    secondary = None
    if world == 1 and not args.no_secondary and args.workload == "ascii4g_lev_m20_k2":
        secondary = run_secondary(F, hs, alphabet, seed, peak)  # (plants more patterns into hs: keep it last)
    filt = float(np.mean(filt_ms))
    achieved = (bhi - blo) / (filt * 1e-3) / 1e9 if filt > 0 else 0.0
    traffic = ncu_traffic()
    line = {"metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak" if kind != "batch" else "strong", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic", "config": config, "matches_per_step": int(nfinal), "wall_ms_per_step": wall_ms / args.steps,
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": ({"lev": "k_filter_sampled" if len(alphabet) > 16 else "k_filter_dense",
                                     "ham": "k_hamming_count"}.get(kind, "all scans of the batch")),
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "peak_source": peak_src, "kernel_ms": filt,
                         "algorithmic_bytes_per_launch": bhi - blo,
                         "traffic": (traffic or {}).get("dram_bytes_per_launch") if (kind == "lev" and len(alphabet) > 16) else None,
                         "traffic_source": "profiles/filter_traffic.json (ncu --set full capture of this kernel; a constant, not "
                                           "measured in this run)"},
            "clocks": clocks}
    if secondary is not None:
        line["secondary"] = secondary
    if parity is not None:
        line["parity"] = parity
    if e2e is not None:
        line["e2e"] = e2e
    if kind == "batch":
        line["config"]["patterns"] = 1024
        line["pattern_GB_per_s"] = value * 1024
    if not args.no_cpu_baseline and world == 1 and reference_available() and kind != "batch":
        # run in a fresh process: the reference arm forks worker processes, which must not inherit
        # this process's CUDA context
        def ref_run(extra):
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload",
                                  args.workload, "--steps", "5", "--warmup", "1"] + extra,
                                 capture_output=True, text=True, timeout=900)
            return json.loads(out.stdout.strip().splitlines()[-1])
        try:
            sample_mib = args.cpu_sample_mib or min(per_gpu >> 20, 1024)
            allc = ref_run(["--cpu-sample-mib", str(sample_mib)])
            line["cpu_baseline"] = dict(allc["cpu_baseline"], matches=allc.get("matches"))
        except Exception as e:  # noqa: BLE001 -- the GPU line must still be printed
            line["cpu_baseline"] = {"error": repr(e)[:200]}
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
