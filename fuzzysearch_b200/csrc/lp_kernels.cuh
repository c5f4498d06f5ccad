// lp_kernels.cuh -- the "linear programming" NFA routes and the generic (per-operation-limit) search.
//
// Both reference NFAs keep a list of candidates that never interact (SURVEY F12), so the search
// decomposes by START POSITION: one thread simulates the candidates born at one start, statement
// by statement as the reference does (duplicate candidates are kept as separate list entries, so
// the raw output is the reference's multiset, not merely its set).  The two candidate lists of a
// thread live in a global scratch slab (cap entries each); an overflow sets CNT_OVERFLOW and the
// host retries with a larger slab.
//
//   k_lev_lp            levenshtein.py:52-148   (route L = m//(k+1) < 3)
//   k_generic_lp        generic_search.py:57-177 over the whole sequence
//   k_verify_generic    generic_search.py:198-237: per n-gram hit, the same NFA on the clipped
//                       window H[max(0,p0-k) : min(N,p0+m+k)] (window end acts as end of input)
#pragma once
#include "kernels.cuh"

namespace fzb {


// ---- Levenshtein LP ------------------------------------------------------------------------------
// candidate = (subseq_index j, dist d) packed j | d<<16
__device__ __forceinline__ bool lp_push(uint32_t *list, int &n, int cap, int j, int d) {
    if (n >= cap) return false;
    list[n++] = (uint32_t)j | ((uint32_t)d << 16);
    return true;
}

// Simulates the candidates whose start is `start` (global).  Returns false on list overflow.
// H[g] must be the haystack byte at global position g (global memory or a staged tile).
// PT: anything with m, k, N (ScanParams, or the per-survivor context of the batch kernels); `tag` goes into the
// records' n-gram field (1 = multiplicity; batches add the pattern number << 8).
template <class PT>
__device__ bool sim_lev_lp(const PT &p, const uint8_t *sP, const uint8_t *H, int64_t start, uint32_t *A,
                           uint32_t *B, int cap, RawRec *out, uint32_t ocap, uint32_t *counters, int tag = 1) {
    const int m = p.m, k = p.k;
    const int64_t N = p.N;
    int nA = 0;
    {
        const uint8_t ch = H[start];
        // make_char2first_subseq_index (levenshtein.py:44-49): first index of ch in P[:k+1]
        int j0 = -1;
        const int lim = min(k, m - 1);
        for (int j = 0; j <= lim; j++)
            if (sP[j] == ch) {
                j0 = j;
                break;
            }
        if (j0 < 0) return true;  // :76-77
        if (j0 + 1 == m) {        // :78-79
            emit(out, ocap, counters, start, start + 1, start, j0, tag);
            return true;
        }
        A[0] = (uint32_t)(j0 + 1) | ((uint32_t)j0 << 16);  // :80-81
        nA = 1;
    }
    int64_t i = start + 1;
    for (; i < N && nA > 0; i++) {  // :73
        const uint8_t ch = H[i];
        int nB = 0;
        for (int c = 0; c < nA; c++) {  // :83
            const int j = (int)(A[c] & 0xFFFFu), d = (int)(A[c] >> 16);
            if (sP[j] == ch) {  // :85
                if (j + 1 == m)
                    emit(out, ocap, counters, start, i + 1, start, d, tag);  // :87-88
                else if (!lp_push(B, nB, cap, j + 1, d))                  // :90-93
                    return false;
            } else {
                if (d == k) continue;                                 // :100-101
                if (!lp_push(B, nB, cap, j, d + 1)) return false;     // :104
                if (i + 1 < N && j + 1 < m)                           // :106
                    if (!lp_push(B, nB, cap, j + 1, d + 1)) return false;  // :109-112
                for (int t = 1; t <= k - d; t++) {                    // :115
                    if (j + t == m) {                                 // :118
                        emit(out, ocap, counters, start, i + 1, start, d + t, tag);
                        break;
                    } else if (sP[j + t] == ch) {  // :126
                        if (j + t + 1 == m)        // :129
                            emit(out, ocap, counters, start, i + 1, start, d + t, tag);
                        else if (!lp_push(B, nB, cap, j + 1 + t, d + t))  // :135-138
                            return false;
                        break;
                    }
                }
            }
        }
        uint32_t *T = A;  // :143
        A = B;
        B = T;
        nA = nB;
    }
    if (i >= N) {  // reached the end of the sequence with live candidates (:145-148)
        for (int c = 0; c < nA; c++) {
            const int j = (int)(A[c] & 0xFFFFu), d = (int)(A[c] >> 16);
            const int dist = d + m - j;
            if (dist <= k) emit(out, ocap, counters, start, N, start, dist, tag);
        }
    }
    return true;
}

constexpr int kLpThreads = 256;  // 4 CTAs per SM: 32 warps hide the shared-memory latency of the tile passes

// One CTA works on tiles of kLpTile start positions: the tile (+ the m+k bytes a candidate can run
// ahead) is staged in shared memory with coalesced loads; phase 1 discards the starts that cannot produce a
// match and queues the survivors; phase 2 hands the queued starts to the threads one by one, so the
// expensive candidate simulation runs with every lane busy.  Phase 1 applies two NECESSARY conditions:
//   (a) the reference only opens a candidate on a character of P[:k+1] (levenshtein.py:44-49,75-80);
//   (b) counting: a raw match (s, e, d <= k) aligns at least m - d pattern characters with EQUAL text
//       characters (every pattern character is matched, substituted or deleted) and spans e - s <= m + k text
//       characters, so the window H[s : s+m+k) must hold at least m - k characters that occur in P at all.
//       A prefix count over the tile makes that one subtraction per start.  On text (95 symbols) (a) keeps
//       ~5 % of the starts and (a)+(b) ~0.1 %: the simulation, which round 1 ran on every (a)-survivor
//       (~70 ms per pattern on 4 GiB), becomes a small tail of an HBM-paced scan.
// Both conditions only DROP starts whose simulation would emit nothing, so the raw multiset is unchanged.
constexpr int kLpTile = 8192;
constexpr int kLpHalo = 2 * kMaxPattern + 16;

// Exclusive prefix counts of class[text[i]] over nchars characters into cnt[0..nchars]; all threads call.
__device__ __forceinline__ void lp_prefix_counts(const uint8_t *text, int nchars, const uint8_t *cls, uint16_t *cnt,
                                                 uint32_t *warp_tot) {
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int per = (nchars + kLpThreads - 1) / kLpThreads;
    const int lo = min(tid * per, nchars), hi = min(lo + per, nchars);
    uint32_t mine = 0;
    for (int i = lo; i < hi; i++) mine += cls[text[i]];
    uint32_t inc = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) warp_tot[w] = inc;
    __syncthreads();
    uint32_t base = inc - mine;
    for (int i = 0; i < w; i++) base += warp_tot[i];
    for (int i = lo; i < hi; i++) {
        cnt[i] = (uint16_t)base;
        base += cls[text[i]];
    }
    if (hi == nchars && lo <= nchars) cnt[nchars] = (uint16_t)base;  // (several threads may write the same total)
    __syncthreads();
}

__global__ void __launch_bounds__(kLpThreads)
k_lev_lp(const ScanParams p, uint32_t *scratch, int cap, RawRec *out, uint32_t ocap, uint32_t *counters) {
    __shared__ uint8_t sP[256];
    __shared__ int16_t sFirst[256];
    __shared__ uint8_t sClass[256];
    __shared__ __align__(16) uint8_t sH[kLpTile + kLpHalo];
    __shared__ uint16_t sCnt[kLpTile + kLpHalo + 2];
    __shared__ uint16_t sQueue[kLpTile];
    __shared__ uint32_t sQn;
    __shared__ uint32_t sWarpTot[kLpThreads / 32];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        sP[i] = p.P[i];
        sFirst[i] = -1;
        sClass[i] = 0;
    }
    __syncthreads();
    if (threadIdx.x == 0) {  // make_char2first_subseq_index: first index of each char within P[:k+1]
        for (int j = min(p.k, p.m - 1); j >= 0; j--) sFirst[p.P[j]] = (int16_t)j;
        for (int j = 0; j < p.m; j++) sClass[p.P[j]] = 1;
    }
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    uint32_t *A = scratch + tid * 2 * (int64_t)cap, *B = A + cap;
    if (p.k >= p.m) {  // levenshtein.py:62-65: an empty match (i,i,m) at every index 0..N
        const int64_t hi = (p.own_hi == p.N) ? p.N + 1 : p.own_hi;
        for (int64_t i = p.own_lo + tid; i < hi; i += stride) emit(out, ocap, counters, i, i, i, p.m, 1);
        return;
    }
    const int64_t hi = min(p.own_hi, p.N);
    const int ahead = p.m + p.k + 1;
    const int win = p.m + p.k, need = p.m - p.k;
    for (int64_t tile_lo = p.own_lo + (int64_t)blockIdx.x * kLpTile; tile_lo < hi; tile_lo += (int64_t)gridDim.x * kLpTile) {
        const int tile_n = (int)min((int64_t)kLpTile, hi - tile_lo);
        const int64_t load_hi = min(min(tile_lo + tile_n + ahead, p.N), p.buf_lo + p.buf_len);
        const int nload = (int)(load_hi - tile_lo);
        const int nwords = (nload + 3) >> 2;  // tile_lo is a multiple of 16: aligned words
        const uint32_t *src = reinterpret_cast<const uint32_t *>(p.H + (tile_lo - p.buf_lo));
        __syncthreads();  // previous tile fully consumed (also orders sFirst / sClass on the first pass)
        for (int w = threadIdx.x; w < nwords; w += blockDim.x) reinterpret_cast<uint32_t *>(sH)[w] = __ldg(src + w);
        if (threadIdx.x == 0) sQn = 0;
        __syncthreads();
        lp_prefix_counts(sH, nload, sClass, sCnt, sWarpTot);
        for (int i = threadIdx.x; i < tile_n; i += blockDim.x)
            if (sFirst[sH[i]] >= 0 && (int)sCnt[min(i + win, nload)] - (int)sCnt[i] >= need)
                sQueue[atomicAdd(&sQn, 1u)] = (uint16_t)i;
        __syncthreads();
        const uint32_t qn = sQn;
        const uint8_t *W = sH - tile_lo;  // W[g]: byte at global position g
        for (uint32_t q = threadIdx.x; q < qn; q += blockDim.x)
            if (!sim_lev_lp(p, sP, W, tile_lo + sQueue[q], A, B, cap, out, ocap, counters))
                atomicExch(&counters[CNT_OVERFLOW], 1u);
    }
}

// ---- streaming form of the Levenshtein LP search -------------------------------------------------------------
// k_lp_scan streams the haystack like the n-gram filters do (coalesced 16-byte loads, every byte read once) and
// applies conditions (a) and (b) of k_lev_lp with bit masks instead of per-tile prefix sums: each lane turns its 16
// bytes into two 16-bit masks through a 256-byte table (bit 0: the byte occurs in P; bit 1: it occurs in P[:k+1]),
// fetches the masks of the next three lanes by shuffle and tests popc(window of m+k bits) >= m-k at the few starts
// whose first-character bit is set.  A warp covers 512 bytes and emits the starts of the first 464 (lanes 29-31
// only supply the look-ahead), survivors are buffered per CTA in shared memory and flushed to a global list with
// one atomic per ~1000 of them.  k_lp_verify then takes ONE SURVIVOR PER THREAD: the bit-parallel automaton
// (SURVEY appendix A.2: state "next pattern index j at cost d" <-> bit j of R[d]; sets instead of the reference's
// candidate lists, so it answers "does this start accept at all?" exactly) discards the starts that emit nothing,
// and the literal simulation (sim_lev_lp: keeps the reference's duplicate candidates, hence its raw multiset) runs
// on the rest.  4 GiB of text, m = 8..14, k = 2..4: ~1 ms per pattern instead of 15 (tile kernel) / 70 (round 1).
constexpr int kLpsThreads = 256;
constexpr int kLpsWarpBytes = 464;                                  // starts a warp emits per iteration (29 lanes)
constexpr int kLpsCtaBytes = (kLpsThreads / 32) * kLpsWarpBytes;    // 3712
constexpr int kLpsFlush = 1024;
constexpr int kLpsBuf = kLpsFlush + kLpsCtaBytes;
constexpr int kLpsMaxWin = 48;                                      // m + k: 15 + 48 <= 63 bits of look-ahead
enum { CNT_LPLIST = 7, CNT_LPWORK = 8 };                            // (the hit-list slots of the dense route)

__global__ void __launch_bounds__(kLpsThreads)
k_lp_scan(const ScanParams p, unsigned long long *list, uint32_t list_cap) {
    __shared__ uint8_t lut[256];
    __shared__ unsigned long long sBuf[kLpsBuf];
    __shared__ uint32_t sN, sBase;
    for (int i = threadIdx.x; i < 256; i += blockDim.x) lut[i] = 0;
    if (threadIdx.x == 0) sN = 0;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int j = 0; j < p.m; j++) lut[p.P[j]] |= 1;
        for (int j = 0; j <= min(p.k, p.m - 1); j++) lut[p.P[j]] |= 2;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int win = p.m + p.k, need = p.m - p.k;
    const unsigned long long wmask = (1ull << win) - 1ull;
    const int64_t hi = min(p.own_hi, p.N);                       // starts are < hi
    const int64_t lim = min(p.N, p.buf_lo + p.buf_len);          // bytes at or beyond this count as "not in P"
    const int64_t base = p.own_lo & ~(int64_t)15;
    const int64_t niter = hi > base ? (hi - base + kLpsCtaBytes - 1) / kLpsCtaBytes : 0;
    for (int64_t it = blockIdx.x; it < niter; it += gridDim.x) {
        const int64_t g0 = base + it * kLpsCtaBytes + (int64_t)warp * kLpsWarpBytes + 16 * lane;  // my 16 bytes
        uint4 d = make_uint4(0, 0, 0, 0);
        if (g0 < lim) d = __ldg(reinterpret_cast<const uint4 *>(p.H + (g0 - p.buf_lo)));  // padded buffer; g0 % 16 == 0
        const uint32_t ws[4] = {d.x, d.y, d.z, d.w};
        uint32_t A = 0, Fm = 0;
#pragma unroll
        for (int i = 0; i < 16; i++) {
            const uint32_t v = lut[(ws[i >> 2] >> (8 * (i & 3))) & 0xFFu];
            A |= (v & 1u) << i;
            Fm |= (v >> 1) << i;
        }
        const int64_t nvalid = lim - g0;  // bytes of mine inside the sequence
        if (nvalid < 16) {
            const uint32_t keep = nvalid <= 0 ? 0u : ((1u << nvalid) - 1u);
            A &= keep;
            Fm &= keep;
        }
        const uint32_t n1 = __shfl_down_sync(0xFFFFFFFFu, A, 1), n2 = __shfl_down_sync(0xFFFFFFFFu, A, 2),
                       n3 = __shfl_down_sync(0xFFFFFFFFu, A, 3);
        const unsigned long long look = (unsigned long long)A | ((unsigned long long)n1 << 16) |
                                        ((unsigned long long)n2 << 32) | ((unsigned long long)n3 << 48);
        if (lane >= 29) Fm = 0;  // look-ahead lanes: the next warp / iteration owns these starts
        bool full = false;
        while (Fm) {
            const int i = __ffs(Fm) - 1;
            Fm &= Fm - 1;
            const int64_t s0 = g0 + i;
            if (s0 < p.own_lo || s0 >= hi) continue;
            if (__popcll((look >> i) & wmask) >= need) {
                const uint32_t slot = atomicAdd(&sN, 1u);
                sBuf[slot] = (unsigned long long)s0;
                full |= slot + 1u >= (uint32_t)kLpsFlush;
            }
        }
        // Flush once the buffer has reached the threshold.  The decision is reduced INSIDE the barrier from what
        // each thread saw before it: a count read after the barrier could already include appends of warps that are
        // an iteration ahead, and the warps of the CTA must agree both on taking this branch (it contains barriers)
        // and on n.  Inside the branch nobody appends, so sN is stable.
        if (__syncthreads_or(full)) {
            const uint32_t n = sN;
            if (threadIdx.x == 0) sBase = atomicAdd(&p.counters[CNT_LPLIST], n);
            __syncthreads();
            const uint32_t b0 = sBase;
            for (uint32_t i = threadIdx.x; i < n; i += blockDim.x)
                if (b0 + i < list_cap) list[b0 + i] = sBuf[i];
            __syncthreads();
            if (threadIdx.x == 0) sN = 0;
            __syncthreads();
        }
    }
    __syncthreads();
    const uint32_t n = sN;
    if (n) {
        if (threadIdx.x == 0) sBase = atomicAdd(&p.counters[CNT_LPLIST], n);
        __syncthreads();
        const uint32_t b0 = sBase;
        for (uint32_t i = threadIdx.x; i < n; i += blockDim.x)
            if (b0 + i < list_cap) list[b0 + i] = sBuf[i];
    }
}

// Does the candidate born at `start` accept anywhere?  (see the header comment above; m <= 31, k <= K)
// One step of the automaton on the match mask M of the next text character: returns 1 if some state accepts, else 0
// and sets `alive`.  (SURVEY appendix A.2; line numbers are levenshtein.py's.)
template <int K>
__device__ __forceinline__ int lp_nfa_step(uint32_t (&R)[K + 1], uint32_t M, bool can_sub, int m, int k, bool &alive) {
    const uint32_t last = 1u << (m - 1), full = (1u << m) - 1u;
    uint32_t nR[K + 1];
#pragma unroll
    for (int d = 0; d <= K; d++) nR[d] = 0;
#pragma unroll
    for (int d = 0; d <= K; d++) {
        const uint32_t r = R[d];
        if (d > k || !r) continue;
        const uint32_t adv = r & M;  // :85-93: a matching character only advances
        if (adv & last) return 1;
        nR[d] |= adv << 1;
        if (d < k) {  // :100-101
            const uint32_t mis = r & ~M;
            if (d + 1 <= K) {
                nR[d + 1] |= mis;                                // insertion (:104)
                if (can_sub) nR[d + 1] |= (mis & ~last) << 1;    // substitution (:106-112)
            }
            uint32_t u = mis;  // deletions, first rule that fires wins per state (:115-138)
#pragma unroll
            for (int t = 1; t <= K; t++) {
                if (t > k - d || !u || t > m) continue;
                if (u & (1u << (m - t))) return 1;     // j + t == m
                const uint32_t hit = u & (M >> t);     // P[j+t] == c
                if (hit) {
                    const uint32_t moved = hit << (t + 1);
                    if (moved & (1u << m)) return 1;     // j + t + 1 == m
                    if (d + t <= K) nR[d + t] |= moved;
                    u &= ~hit;
                }
            }
        }
    }
    uint32_t any = 0;
#pragma unroll
    for (int d = 0; d <= K; d++) {
        R[d] = nR[d] & full;
        any |= R[d];
    }
    alive = any != 0;
    return 0;
}

// live states at the end of the sequence accept iff d + m - j <= k (:145-148)
template <int K>
__device__ __forceinline__ bool lp_nfa_end(const uint32_t (&R)[K + 1], int m, int k) {
#pragma unroll
    for (int d = 0; d <= K; d++) {
        if (d > k) continue;
        uint32_t r = R[d];
        while (r) {
            const int j = __ffs(r) - 1;
            r &= r - 1;
            if (d + m - j <= k) return true;
        }
    }
    return false;
}

// Does the candidate born at `start` accept anywhere?  sPM32: the pattern's 256 match masks (shared or global).
template <int K>
__device__ __forceinline__ bool lp_nfa_any(const uint32_t *sPM32, const uint8_t *H, int64_t start, int64_t N, int m,
                                           int k, int j0) {
    if (j0 + 1 == m) return true;  // levenshtein.py:78-79
    uint32_t R[K + 1];
#pragma unroll
    for (int d = 0; d <= K; d++) R[d] = (d == j0) ? (1u << (j0 + 1)) : 0u;  // :80-81
    for (int64_t i = start + 1; i < N; i++) {
        bool alive = true;
        if (lp_nfa_step<K>(R, sPM32[H[i]], i + 1 < N, m, k, alive)) return true;
        if (!alive) return false;
    }
    return lp_nfa_end<K>(R, m, k);
}

__global__ void __launch_bounds__(kLpThreads)
k_lp_verify(const ScanParams p, const unsigned long long *list, uint32_t list_cap, uint32_t *scratch, int cap,
            RawRec *out, uint32_t ocap, uint32_t *counters) {
    __shared__ uint8_t sP[256];
    __shared__ int16_t sFirst[256];
    __shared__ uint32_t sPM32[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        sP[i] = p.P[i];
        sFirst[i] = -1;
        uint32_t v = 0;
        for (int j = 0; j < p.m && j < 32; j++) v |= (uint32_t)(p.P[j] == i) << j;
        sPM32[i] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0)
        for (int j = min(p.k, p.m - 1); j >= 0; j--) sFirst[p.P[j]] = (int16_t)j;
    __syncthreads();
    const uint32_t n = counters[CNT_LPLIST];
    if (n > list_cap) {  // the list overflowed: the host repeats the search with the tile kernel
        if (blockIdx.x == 0 && threadIdx.x == 0) counters[CNT_LPWORK] = 1;
        return;
    }
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t *A = scratch + tid * 2 * (int64_t)cap, *B = A + cap;
    const uint8_t *W = p.H - p.buf_lo;  // W[g]: byte at global position g
    const bool use_nfa = p.m <= 31 && p.k <= 8;
    for (int64_t i = tid; i < (int64_t)n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t st = (int64_t)list[i];
        if (use_nfa) {
            const int j0 = sFirst[W[st]];
            const bool any = p.k <= 4 ? lp_nfa_any<4>(sPM32, W, st, p.N, p.m, p.k, j0)
                                      : lp_nfa_any<8>(sPM32, W, st, p.N, p.m, p.k, j0);
            if (!any) continue;
        }
        if (!sim_lev_lp(p, sP, W, st, A, B, cap, out, ocap, counters)) atomicExch(&counters[CNT_OVERFLOW], 1u);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&counters[CNT_CAND], n);
}

// ---- generic NFA ---------------------------------------------------------------------------------
// candidate = (subseq_index j, l_dist, n_subs, n_ins, n_dels) packed 8|6|6|6|6 bits
__device__ __forceinline__ uint32_t gpack(int j, int l, int ns, int ni, int nd) {
    return (uint32_t)j | ((uint32_t)l << 8) | ((uint32_t)ns << 14) | ((uint32_t)ni << 20) | ((uint32_t)nd << 26);
}
__device__ __forceinline__ bool g_push(uint32_t *list, int &n, int cap, uint32_t v) {
    if (n >= cap) return false;
    list[n++] = v;
    return true;
}

// Candidates born at `start`, over the sequence that ends (exclusive) at `seq_end` (both global).
// anchor_idx / anchor_ngram tag the emitted records (n-gram hit that opened the window, or start).
// H[g] must be the haystack byte at global position g (global memory, or the staged window).
// PT: ScanParams, or the per-segment context of seg_kernels.cuh (anything with m, k, max_subs, max_ins, max_dels).
template <class PT>
__device__ bool sim_generic(const PT &p, const uint8_t *sP, const uint8_t *H, int64_t start,
                            int64_t seq_end, uint32_t *A, uint32_t *B, int cap, int64_t anchor_idx,
                            int anchor_ngram, RawRec *out, uint32_t ocap, uint32_t *counters) {
    const int m = p.m, max_l = p.k, max_subs = p.max_subs, max_ins = p.max_ins, max_dels = p.max_dels;
    A[0] = gpack(0, 0, 0, 0, 0);  // generic_search.py:81
    int nA = 1;
    int64_t i = start;
    for (; i < seq_end && nA > 0; i++) {  // :79
        const uint8_t ch = H[i];
        int nB = 0;
        for (int c = 0; c < nA; c++) {  // :84
            const uint32_t v = A[c];
            const int j = (int)(v & 0xFFu), l = (int)((v >> 8) & 63u), ns = (int)((v >> 14) & 63u),
                      ni = (int)((v >> 20) & 63u), nd = (int)((v >> 26) & 63u);
            if (ch == sP[j]) {  // :86
                if (j + 1 == m)
                    emit(out, ocap, counters, start, i + 1, anchor_idx, l, anchor_ngram);  // :88-89
                else if (!g_push(B, nB, cap, gpack(j + 1, l, ns, ni, nd)))                // :91-94
                    return false;
            } else {
                if (l == max_l) continue;  // :101-102
                if (ni < max_ins)          // :104-109
                    if (!g_push(B, nB, cap, gpack(j, l + 1, ns, ni + 1, nd))) return false;
                if (j + 1 < m) {            // :111
                    if (ns < max_subs) {    // :112-119
                        if (!g_push(B, nB, cap, gpack(j + 1, l + 1, ns + 1, ni, nd))) return false;
                    } else if (nd < max_dels && ni < max_ins) {  // :120-128
                        if (!g_push(B, nB, cap, gpack(j + 1, l + 1, ns, ni + 1, nd + 1))) return false;
                    }
                } else {  // :129-138
                    if (ns < max_subs || (nd < max_dels && ni < max_ins))
                        emit(out, ocap, counters, start, i + 1, anchor_idx, l + 1, anchor_ngram);
                }
                const int lim = min(max_dels - nd, max_l - l);  // :141
                for (int t = 1; t <= lim; t++) {
                    if (j + t == m) {  // :144-147  (end excludes the current char)
                        emit(out, ocap, counters, start, i, anchor_idx, l + t, anchor_ngram);
                        break;
                    } else if (sP[j + t] == ch) {  // :151
                        if (j + t + 1 == m)        // :154-156
                            emit(out, ocap, counters, start, i, anchor_idx, l + t, anchor_ngram);
                        else if (!g_push(B, nB, cap, gpack(j + 1 + t, l + t, ns, ni, nd + t)))  // :159-164
                            return false;
                        break;
                    }
                }
            }
        }
        uint32_t *T = A;  // :170
        A = B;
        B = T;
        nA = nB;
    }
    if (i >= seq_end) {  // :172-177
        for (int c = 0; c < nA; c++) {
            const uint32_t v = A[c];
            const int j = (int)(v & 0xFFu), l = (int)((v >> 8) & 63u), nd = (int)((v >> 26) & 63u);
            const int t = m - j;
            if (nd + t <= max_dels && l + t <= max_l)
                emit(out, ocap, counters, start, seq_end, anchor_idx, l + t, anchor_ngram);
        }
    }
    return true;
}

// Same tile scheme as k_lev_lp.  The generic NFA opens a candidate at EVERY index (generic_search.py:81), so
// only the counting condition applies: a match costs l <= max_l, every pattern character it does not align with
// an equal text character costs at least 1 (substitution, deletion, or the insertion+deletion pair of
// :120-128), and it consumes at most m + max_l text characters -- so H[s : s+m+max_l) must hold at least
// m - max_l characters that occur in the pattern.
__global__ void __launch_bounds__(kLpThreads)
k_generic_lp(const ScanParams p, uint32_t *scratch, int cap, RawRec *out, uint32_t ocap, uint32_t *counters) {
    __shared__ uint8_t sP[256];
    __shared__ uint8_t sClass[256];
    __shared__ __align__(16) uint8_t sH[kLpTile + kLpHalo];
    __shared__ uint16_t sCnt[kLpTile + kLpHalo + 2];
    __shared__ uint16_t sQueue[kLpTile];
    __shared__ uint32_t sQn;
    __shared__ uint32_t sWarpTot[kLpThreads / 32];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        sP[i] = p.P[i];
        sClass[i] = 0;
    }
    __syncthreads();
    if (threadIdx.x == 0)
        for (int j = 0; j < p.m; j++) sClass[p.P[j]] = 1;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t *A = scratch + tid * 2 * (int64_t)cap, *B = A + cap;
    const int64_t hi = min(p.own_hi, p.N);
    const int ahead = p.m + p.k + 1;
    const int win = p.m + p.k, need = p.m - p.k;  // p.k = max_l
    for (int64_t tile_lo = p.own_lo + (int64_t)blockIdx.x * kLpTile; tile_lo < hi; tile_lo += (int64_t)gridDim.x * kLpTile) {
        const int tile_n = (int)min((int64_t)kLpTile, hi - tile_lo);
        const int64_t load_hi = min(min(tile_lo + tile_n + ahead, p.N), p.buf_lo + p.buf_len);
        const int nload = (int)(load_hi - tile_lo);
        const int nwords = (nload + 3) >> 2;
        const uint32_t *src = reinterpret_cast<const uint32_t *>(p.H + (tile_lo - p.buf_lo));
        __syncthreads();
        for (int w = threadIdx.x; w < nwords; w += blockDim.x) reinterpret_cast<uint32_t *>(sH)[w] = __ldg(src + w);
        if (threadIdx.x == 0) sQn = 0;
        __syncthreads();
        lp_prefix_counts(sH, nload, sClass, sCnt, sWarpTot);
        for (int i = threadIdx.x; i < tile_n; i += blockDim.x)
            if ((int)sCnt[min(i + win, nload)] - (int)sCnt[i] >= need) sQueue[atomicAdd(&sQn, 1u)] = (uint16_t)i;
        __syncthreads();
        const uint32_t qn = sQn;
        const uint8_t *W = sH - tile_lo;  // W[g]: byte at global position g
        for (uint32_t q = threadIdx.x; q < qn; q += blockDim.x) {
            const int64_t st = tile_lo + sQueue[q];
            if (!sim_generic(p, sP, W, st, p.N, A, B, cap, st, 1, out, ocap, counters))
                atomicExch(&counters[CNT_OVERFLOW], 1u);
        }
    }
}

// Generic n-gram route: one warp per marked granule.  Phase 1: lane <-> anchor position, exact
// n-gram test (generic_search.py:221-227).  Phase 2: for every hit, the lanes of the warp split
// the starts of the clipped window (:229-237) and run the NFA.
__global__ void __launch_bounds__(kLpThreads)
k_verify_generic(const ScanParams p, uint64_t bitmap_words, uint32_t *scratch, int cap, RawRec *out,
                 uint32_t ocap, uint32_t *counters) {
    __shared__ uint8_t sP[256];
    __shared__ uint32_t sWinAll[kLpThreads / 32][kWinWords];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) sP[i] = p.P[i];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    uint32_t *sWin = sWinAll[threadIdx.x >> 5];
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t *A = scratch + tid * 2 * (int64_t)cap, *B = A + cap;
    const uint64_t gwarp = (uint64_t)tid >> 5;
    const uint64_t nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const int m = p.m, k = p.k, L = p.L;
    const int64_t N = p.N;
    for (uint64_t wbase = gwarp * 32; wbase < bitmap_words; wbase += nwarps * 32) {
        const uint64_t wi = wbase + lane;
        uint32_t bits = wi < bitmap_words ? p.bitmap[wi] : 0u;
        if (bits) p.bitmap[wi] = 0u;  // consumed: the bitmap is all-zero again when the kernel ends
        unsigned active = __ballot_sync(0xFFFFFFFFu, bits != 0);
        while (active) {
            const int src = __ffs(active) - 1;
            active &= active - 1;
            uint32_t b = __shfl_sync(0xFFFFFFFFu, bits, src);
            if (lane == 0) atomicAdd(&counters[CNT_CAND], (uint32_t)__popc(b));
            while (b) {
                const int bit = __ffs(b) - 1;
                b &= b - 1;
                const int64_t gbase = p.buf_lo + (((int64_t)(wbase + src) * 32 + bit) << kGranuleShift);
                const int64_t alo = stage_window(p, gbase, m + k, lane, sWin);
                const uint8_t *W = reinterpret_cast<const uint8_t *>(sWin) - alo;  // W[g]: byte at global g
                for (int half = 0; half < kGranule / 32; half++) {
                    const int64_t idx = gbase + half * 32 + lane;
                    const bool owned = idx >= p.own_lo && idx < p.own_hi;
                    for (int j = 0; j < p.n_ngrams; j++) {
                        const int s = j * L;
                        bool hit = false;
                        if (owned) {
                            int64_t ws = max((int64_t)0, (int64_t)(s - k));  // :223
                            int64_t we = min(N, N - m + s + L + k);          // :224
                            if (we > ws) {                                   // :225-226
                                ws = max((int64_t)0, min(ws, N));
                                we = max(ws, min(we, N));
                                if (idx >= ws && idx + L <= we) {
                                    const uint8_t *h = W + idx;
                                    hit = true;
                                    for (int i = 0; i < L; i++)
                                        if (h[i] != sP[s + i]) {
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
                            const int64_t hidx = gbase + half * 32 + hl;
                            const int64_t p0 = hidx - s;
                            const int64_t wlo = max((int64_t)0, p0 - k);      // :231
                            const int64_t whi = min(N, p0 + m + k);
                            for (int64_t st = wlo + lane; st < whi; st += 32)
                                if (!sim_generic(p, sP, W, st, whi, A, B, cap, hidx, j, out, ocap, counters))
                                    atomicExch(&counters[CNT_OVERFLOW], 1u);
                        }
                    }
                }
            }
        }
    }
}

}  // namespace fzb
