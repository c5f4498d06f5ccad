// seg_kernels.cuh -- one pattern over MANY short sequences (segments of one resident buffer) in one device pass.
//
// A caller with 10^6 reads of a few hundred bytes would otherwise pay the whole fixed cost of a search (upload,
// three or four launches, a synchronisation, a copy) per read.  Here the reads are packed back to back into one
// buffer, `offsets[count + 1]` delimits them, and every segment is searched AS IF IT WERE THE WHOLE SEQUENCE:
// window clipping at 0 and at the segment's own length, positions segment-local.
//
//   k_seg_search   one warp per segment (atomic work counter).  The segment (<= kSegMaxBytes) is staged in the warp's
//                  shared window; the lanes walk its anchors / starts 32 at a time and call the device routines of
//                  the single-sequence routes with a per-segment context (N = segment length, own = [0, N)):
//                  verify_anchor_lev on every anchor (it tests n-gram occurrence and window itself, so testing every
//                  anchor is exact), sim_lev_lp / sim_generic on every start, the generic n-gram window NFA, and the
//                  plain Hamming / exact comparison.  The segment number travels in the records' n-gram field
//                  (seg << 8 | what the route puts there), as the batch kernels carry the pattern number.
//   k_seg_hist     raw records per segment
//   k_seg_scan     exclusive scan of those counts (one CTA)
//   k_seg_scatter  counting sort: the canonical keys of the records, grouped by segment
//   k_seg_post     one warp per non-empty segment: sorts the segment's keys and runs the sweep of k_post (running
//                  hull maximum, a new group iff start >= hull, winner = min (dist, -(end-start)), ties -> smallest
//                  (start, end)).  Sorted raw keys and final keys go straight into mapped host memory.  A segment
//                  with more than kSegPostMax raw records is left unsorted and flagged; the host consolidates it.
// Segments longer than kSegMaxBytes are skipped here; the host searches each of them with the single-sequence
// entry points (api.cu: fzb_search_segments).
#pragma once
#include "lp_kernels.cuh"
#include "post_kernels.cuh"

namespace fzb {

constexpr int kSegMaxBytes = FZB_SEG_SHORT_BYTES;  // longest segment a warp stages (DESIGN.md 5.8: how it was chosen)
constexpr int kSegThreads = 128;
constexpr int kSegWarps = kSegThreads / 32;
constexpr int kSegWinWords = kSegMaxBytes / 4 + 2;  // + the misalignment of the segment's first byte
constexpr int kSegPostMax = 256;               // raw records of one segment a warp sorts in shared memory
constexpr uint32_t kSegNoFinal = 0xFFFFFFFFu;  // k_seg_post: segment left to the host
enum { SEG_EXACT = 0, SEG_HAMMING = 1, SEG_LEV_NGRAMS = 2, SEG_LEV_LP = 3, SEG_GEN_NGRAMS = 4, SEG_GEN_LP = 5 };

struct SegParams {
    const uint8_t *H;          // the handle's buffer: segment i is H[offsets[i] : offsets[i+1])
    const uint64_t *offsets;   // device copy of offsets[0 .. count]
    uint32_t count;
    int32_t m, k, L, n_ngrams;
    int32_t max_subs, max_ins, max_dels;
    uint32_t *counters;
    uint8_t P[256];
};

// What the shared device routines read of a sequence (verify_anchor_lev, sim_lev_lp, sim_generic): one segment.
struct SegCtx {
    const uint8_t *H;
    int64_t buf_lo, buf_len, N, own_lo, own_hi;
    int32_t m, k, L, n_ngrams;
    int32_t max_subs, max_ins, max_dels;
};

template <int ROUTE, int VM>
__global__ void __launch_bounds__(kSegThreads)
k_seg_search(const SegParams p, uint32_t *scratch, int cap, RawRec *out, uint32_t ocap) {
    __shared__ uint8_t sP[256];
    __shared__ unsigned long long sPM[(ROUTE == SEG_LEV_NGRAMS && VM < 2) ? 256 : 1];
    __shared__ uint32_t sWinAll[kSegWarps][kSegWinWords];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) sP[i] = p.P[i];
    if (ROUTE == SEG_LEV_NGRAMS && VM < 2) build_pm(sPM, p.P, p.m, threadIdx.x, blockDim.x);
    __syncthreads();
    DpHolder<ROUTE == SEG_LEV_NGRAMS ? VM : 0> dp_holder;
    DpScratch *S = dp_holder.get();
    const int lane = threadIdx.x & 31;
    uint32_t *sWin = sWinAll[threadIdx.x >> 5];
    uint32_t *counters = p.counters;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t *A = scratch + tid * 2 * (int64_t)cap, *B = A + cap;  // LP candidate lists (LP / generic routes only)
    const int m = p.m, k = p.k;
    for (;;) {
        uint32_t seg = 0;
        if (lane == 0) seg = atomicAdd(&counters[CNT_WORK], 1u);
        seg = __shfl_sync(0xFFFFFFFFu, seg, 0);
        if (seg >= p.count) break;
        const int64_t lo = (int64_t)p.offsets[seg];
        const int64_t n = (int64_t)p.offsets[seg + 1] - lo;
        if (n > kSegMaxBytes) continue;  // long segment: searched by the host on its own
        const int64_t alo = lo & ~(int64_t)3;
        const int nwords = (int)((lo + n - alo + 3) >> 2);
        const uint32_t *src = reinterpret_cast<const uint32_t *>(p.H + alo);  // padded buffer: reads past the end are safe
        __syncwarp();
        for (int w = lane; w < nwords; w += 32) sWin[w] = __ldg(src + w);
        __syncwarp();
        const uint8_t *W = reinterpret_cast<const uint8_t *>(sWin) + (lo - alo);  // W[g]: byte g of the segment
        const SegCtx c{W, 0, n, n, 0, n, m, k, p.L, p.n_ngrams, p.max_subs, p.max_ins, p.max_dels};
        const int tag = (int)(seg << 8);
        if (ROUTE == SEG_EXACT || ROUTE == SEG_HAMMING) {
            // search_exact.py:45-56 / substitutions_only.py:37-63: every start with room for the whole pattern
            for (int64_t st = lane; st + m <= n; st += 32) {
                int d = 0;
                for (int i = 0; i < m && d <= k; i++) d += W[st + i] != sP[i];
                if (d <= k) emit(out, ocap, counters, st, st + m, st, d, tag);
            }
        } else if (ROUTE == SEG_LEV_NGRAMS) {
            for (int64_t base = 0; base < n; base += 32) {  // (the whole warp: verify_anchor_lev votes)
                const int64_t idx = base + lane;
                verify_anchor_lev<VM>(c, sP, sPM, W, idx, idx < n, S, out, ocap, counters, 0, c.n_ngrams, tag);
            }
        } else if (ROUTE == SEG_LEV_LP) {
            if (k >= m) {  // levenshtein.py:62-65: an empty match (i, i, m) at every index 0..N
                for (int64_t i = lane; i <= n; i += 32) emit(out, ocap, counters, i, i, i, m, tag | 1);
            } else {
                for (int64_t st = lane; st < n; st += 32)
                    if (!sim_lev_lp(c, sP, W, st, A, B, cap, out, ocap, counters, tag | 1))
                        atomicExch(&counters[CNT_OVERFLOW], 1u);
            }
        } else if (ROUTE == SEG_GEN_LP) {
            for (int64_t st = lane; st < n; st += 32)
                if (!sim_generic(c, sP, W, st, n, A, B, cap, st, tag | 1, out, ocap, counters))
                    atomicExch(&counters[CNT_OVERFLOW], 1u);
        } else {  // SEG_GEN_NGRAMS: the per-hit windows of k_verify_generic (generic_search.py:198-237)
            const int L = p.L;
            for (int64_t base = 0; base < n; base += 32) {
                const int64_t idx = base + lane;
                for (int j = 0; j < p.n_ngrams; j++) {
                    const int s = j * L;
                    bool hit = false;
                    if (idx < n) {
                        int64_t ws = max((int64_t)0, (int64_t)(s - k));  // :223
                        int64_t we = min(n, n - m + s + L + k);          // :224
                        if (we > ws) {                                   // :225-226
                            ws = max((int64_t)0, min(ws, n));
                            we = max(ws, min(we, n));
                            if (idx >= ws && idx + L <= we) {
                                hit = true;
                                for (int i = 0; i < L; i++)
                                    if (W[idx + i] != sP[s + i]) {
                                        hit = false;
                                        break;
                                    }
                            }
                        }
                    }
                    unsigned hits = __ballot_sync(0xFFFFFFFFu, hit);
                    while (hits) {
                        const int hl = __ffs(hits) - 1;
                        hits &= hits - 1;
                        const int64_t hidx = base + hl;
                        const int64_t p0 = hidx - s;
                        const int64_t wlo = max((int64_t)0, p0 - k);  // :231
                        const int64_t whi = min(n, p0 + m + k);
                        for (int64_t st = wlo + lane; st < whi; st += 32)
                            if (!sim_generic(c, sP, W, st, whi, A, B, cap, hidx, tag | j, out, ocap, counters))
                                atomicExch(&counters[CNT_OVERFLOW], 1u);
                    }
                }
            }
        }
    }
}

// An attempt whose output or candidate lists overflowed is repeated by the host: the grouping kernels skip it.
__device__ __forceinline__ bool seg_attempt_valid(const uint32_t *counters, uint32_t ocap) {
    return counters[CNT_OUT] <= ocap && counters[CNT_OVERFLOW] == 0;
}

__device__ __forceinline__ uint32_t seg_of(const RawRec &r) { return (uint32_t)r.ngram >> 8; }

constexpr int kSegSortThreads = 256;

__global__ void __launch_bounds__(kSegSortThreads)
k_seg_hist(const RawRec *out, uint32_t ocap, const uint32_t *counters, uint32_t *seg_cnt) {
    if (!seg_attempt_valid(counters, ocap)) return;
    const uint32_t n = counters[CNT_OUT];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        atomicAdd(&seg_cnt[seg_of(out[i])], 1u);
}

// seg_off[s] = sum of seg_cnt[0 .. s), cursor = the same; hdr (mapped host) = record count, overflow flag.
// One CTA of kPostThreads: thread t owns a contiguous run of segments.
__global__ void __launch_bounds__(kPostThreads, 1)
k_seg_scan(const uint32_t *seg_cnt, uint32_t count, const uint32_t *counters, uint32_t ocap, uint32_t *seg_off,
           uint32_t *cursor, uint32_t *h_hdr) {
    __shared__ uint32_t scratch[33];
    if (threadIdx.x == 0) {
        h_hdr[0] = counters[CNT_OUT];
        h_hdr[1] = counters[CNT_OVERFLOW];
    }
    if (!seg_attempt_valid(counters, ocap)) return;
    const uint32_t per = (count + kPostThreads - 1) / kPostThreads;
    const uint32_t lo = min(count, threadIdx.x * per), hi = min(count, lo + per);
    uint32_t mine = 0;
    for (uint32_t s = lo; s < hi; s++) mine += seg_cnt[s];
    uint32_t total;
    uint32_t acc = block_scan_sum(mine, scratch, &total);
    for (uint32_t s = lo; s < hi; s++) {
        seg_off[s] = acc;
        cursor[s] = acc;
        acc += seg_cnt[s];
    }
    if (threadIdx.x == 0) seg_off[count] = total;
}

__global__ void __launch_bounds__(kSegSortThreads)
k_seg_scatter(const RawRec *out, uint32_t ocap, const uint32_t *counters, uint32_t *cursor, uint64_t *keys) {
    if (!seg_attempt_valid(counters, ocap)) return;
    const uint32_t n = counters[CNT_OUT];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const RawRec r = out[i];
        keys[atomicAdd(&cursor[seg_of(r)], 1u)] = canonical_key(r);
    }
}

// Key order is (start, end, dist); the winner of a group minimises (dist, -(end-start)), then (start, end).
__device__ __forceinline__ bool seg_better(uint64_t a, uint64_t b) {
    const uint32_t da = (uint32_t)(a & 0xFFu), db = (uint32_t)(b & 0xFFu);
    if (da != db) return da < db;
    const uint32_t la = (uint32_t)(a >> 8) & 0x3FFu, lb = (uint32_t)(b >> 8) & 0x3FFu;
    if (la != lb) return la > lb;
    return a < b;
}

// One warp per 32 segments: the lanes read 32 counts at once, then the warp takes the non-empty ones in turn.
// seg_nfin[s] = number of final keys of segment s (kSegNoFinal: left to the host); h_raw / h_fin (mapped host)
// hold each segment's keys from seg_off[s] on.
__global__ void __launch_bounds__(kSegThreads)
k_seg_post(const uint32_t *seg_cnt, const uint32_t *seg_off, uint32_t count, const uint64_t *keys,
           const uint32_t *counters, uint32_t ocap, int consolidate, uint32_t *seg_nfin, uint64_t *h_raw,
           uint64_t *h_fin) {
    __shared__ uint64_t sKeys[kSegWarps][kSegPostMax];
    __shared__ uint64_t sSorted[kSegWarps][kSegPostMax];
    if (!seg_attempt_valid(counters, ocap)) return;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    uint64_t *sK = sKeys[wib], *sS = sSorted[wib];
    const uint32_t gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t nwarps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t base = gwarp * 32; base < count; base += nwarps * 32) {
        const uint32_t s = base + lane;
        const uint32_t my_n = s < count ? seg_cnt[s] : 0u;
        const uint32_t my_off = s < count ? seg_off[s] : 0u;
        uint32_t my_fin = 0;
        unsigned todo = __ballot_sync(0xFFFFFFFFu, my_n != 0);
        while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            const uint32_t n = __shfl_sync(0xFFFFFFFFu, my_n, src);
            const uint32_t off = __shfl_sync(0xFFFFFFFFu, my_off, src);
            uint32_t nfin;
            if (n > (uint32_t)kSegPostMax) {
                for (uint32_t i = lane; i < n; i += 32) h_raw[off + i] = keys[off + i];
                nfin = kSegNoFinal;
            } else {
                for (uint32_t i = lane; i < n; i += 32) sK[i] = keys[off + i];
                __syncwarp();
                for (uint32_t i = lane; i < n; i += 32) {  // rank = number of keys before this one (stable)
                    const uint64_t x = sK[i];
                    uint32_t r = 0;
                    for (uint32_t j = 0; j < n; j++) {
                        const uint64_t y = sK[j];
                        r += (y < x) || (y == x && j < i);
                    }
                    sS[r] = x;
                }
                __syncwarp();
                for (uint32_t i = lane; i < n; i += 32) h_raw[off + i] = sS[i];
                nfin = n;
                if (consolidate) {
                    if (lane == 0) {
                        uint64_t best = sS[0];
                        uint64_t hull = (sS[0] >> 18) + ((sS[0] >> 8) & 0x3FFu);
                        uint32_t g = 0;
                        for (uint32_t i = 1; i < n; i++) {
                            const uint64_t x = sS[i];
                            const uint64_t st = x >> 18, en = st + ((x >> 8) & 0x3FFu);
                            if (st < hull) {
                                if (seg_better(x, best)) best = x;
                                hull = max(hull, en);
                            } else {
                                h_fin[off + g++] = best;
                                best = x;
                                hull = en;
                            }
                        }
                        h_fin[off + g++] = best;
                        nfin = g;
                    }
                    nfin = __shfl_sync(0xFFFFFFFFu, nfin, 0);
                }
                __syncwarp();  // sK / sS are reused by the next segment
            }
            if (lane == src) my_fin = nfin;
        }
        if (s < count) seg_nfin[s] = my_fin;
    }
}

}  // namespace fzb
