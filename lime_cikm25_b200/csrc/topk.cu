// Top-k of every user's scores over a news pool (sm_100a).
//
// A recommender serves "which k news of the current pool should user u see": the pool scores of a user are a row of
// up to 2^31 floats, and only k <= 1024 of them leave the device.  lime_rank_metrics' O(C^2) warp ranking is built for
// ~37 candidates; this file selects without ranking the pool.
//
// Key.  Every returnable position c of user u gets a 64-bit key  ord(score) << 32 | ~pool_index[c],  ord an
// order-preserving map of the fp32 score (-0.0 canonicalised to +0.0).  Keys are unique per position (for distinct
// pool_index), so "the k largest keys" is a well-defined set and their descending order is the contract's order:
// score descending, equal scores by ascending pool_index.  NaN, excluded and clicked positions get no key; a key is
// never 0 (ord(-inf) = 0x007fffff), so 0 marks an empty slot.
//
// Rounds.  A CTA owns one group of at most kSliceMax inputs of one user.  It reads each input once, compacts the keys
// into shared memory (warp-aggregated appends), finds the k-th largest key by an MSD radix select over 8-bit digits
// on the resident keys (usually 2-3 digits: it stops as soon as the boundary digit's bin is taken whole), and keeps
// the keys at or above it.  Round 0 reads the scores (groups sized so that about 2 CTAs per SM are busy even for one
// user); a round whose user has more than one group writes its <= k keys per group to scratch and the next round
// selects from groups x k keys (at least 8 groups fold into one, so a 300,000-news pool takes three launches at
// k = 1024).  The last round sorts its <= k keys (bitonic, shared memory) and writes ids and scores.
//
// Clicked exclusion.  Round 0 sorts the user's masked-in history ids (H <= 224) in shared memory once per CTA; every
// position binary-searches its pool_news there.
#include "common.cuh"

namespace lime {

constexpr int kTopkThreads = 512;
constexpr int kSliceMax = 8192;          // keys of one group resident in shared memory (64 KB)
constexpr int kHistMax = 224;            // LimeImpressions.max_history limit of the scoring kernels
__host__ __device__ inline int64_t topk_cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

__device__ __forceinline__ uint32_t score_ord(float s) {
    const uint32_t u = __float_as_uint(s == 0.0f ? 0.0f : s);      // -0.0 == +0.0
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__device__ __forceinline__ float ord_score(uint32_t o) {
    return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}

__device__ __forceinline__ uint64_t pool_key(float s, int32_t pool_index) {
    return ((uint64_t)score_ord(s) << 32) | (uint32_t)~(uint32_t)pool_index;
}

// The masked-in history ids of user u, sorted ascending into hsorted[0, nh); returns nh.  Every thread of a
// kTopkThreads-thread CTA calls (it synchronises); *s_nh must be 0 and visible to all threads on entry.
__device__ __forceinline__ int load_history(const int32_t *__restrict__ hist_news, const uint8_t *__restrict__ hist_mask,
                                            int max_history, int64_t u, int *hraw, int *hsorted, int *s_nh) {
    const int tid = threadIdx.x;
    for (int h0 = 0; h0 < max_history; h0 += kTopkThreads) {       // masked-in ids of the history, then rank-sorted
        const int h = h0 + tid;
        const bool ok = h < max_history && hist_mask[u * max_history + h] != 0;
        const unsigned m = __ballot_sync(0xffffffffu, ok);
        if (m) {
            const int lane = tid & 31, leader = __ffs(m) - 1;
            int base = 0;
            if (lane == leader) base = atomicAdd(s_nh, __popc(m));
            base = __shfl_sync(0xffffffffu, base, leader);
            if (ok) hraw[base + __popc(m & ((1u << lane) - 1u))] = hist_news[u * max_history + h];
        }
    }
    __syncthreads();
    const int nh = *s_nh;
    for (int t = tid; t < nh; t += kTopkThreads) {
        const int v = hraw[t];
        int r = 0;
        for (int j = 0; j < nh; ++j) r += hraw[j] < v || (hraw[j] == v && j < t);
        hsorted[r] = v;
    }
    __syncthreads();
    return nh;
}

// The exclusion test: may pool position i with score s be returned to the user whose sorted history is hsorted[0, nh)?
// Not NaN, not excluded, and its news not clicked (binary search; nh == 0 skips it).
__device__ __forceinline__ bool returnable(float s, int64_t i, const uint8_t *__restrict__ exclude,
                                           const int32_t *__restrict__ pool_news, const int *hsorted, int nh) {
    bool ok = s == s && !(exclude != nullptr && exclude[i]);
    if (ok && nh > 0) {
        const int nw = pool_news[i];
        int a = 0, b = nh;                    // first slot >= nw
        while (a < b) {
            const int mid = (a + b) >> 1;
            if (hsorted[mid] < nw) a = mid + 1; else b = mid;
        }
        ok = !(a < nh && hsorted[a] == nw);
    }
    return ok;
}

// Block-wide append of `key` where `ok`; every lane of the warp must call (the loop bounds below are warp-uniform).
// Appends past `cap` are dropped (only reachable with duplicate pool_index values).
__device__ __forceinline__ void append_key(bool ok, uint64_t key, uint64_t *buf, int *count, int cap) {
    const unsigned m = __ballot_sync(0xffffffffu, ok);
    if (m == 0) return;
    const int lane = threadIdx.x & 31;
    const int leader = __ffs(m) - 1;
    int base = 0;
    if (lane == leader) base = atomicAdd(count, __popc(m));
    base = __shfl_sync(0xffffffffu, base, leader);
    const int pos = base + __popc(m & ((1u << lane) - 1u));
    if (ok && pos < cap) buf[pos] = key;
}

// One round: CTA blockIdx.x = u * groups + g selects the top-k keys of inputs [g * slice, (g + 1) * slice) of user u.
// kScores: inputs are scores [users, n_in] (round 0); otherwise keys [users, n_in] of the previous round (0 = empty).
// keys_out != NULL: write the group's keys unsorted to keys_out[(u * groups + g) * k ..] (0-padded); otherwise this is
// the last round (groups == 1): sort and write out_index / out_score / out_count.
template <bool kScores>
__global__ void __launch_bounds__(kTopkThreads)
pool_topk_kernel(const float *__restrict__ scores, const uint64_t *__restrict__ keys_in, int64_t n_in, int32_t slice,
                 int32_t groups, const int32_t *__restrict__ pool_index, const int32_t *__restrict__ pool_news,
                 const uint8_t *__restrict__ exclude, const int32_t *__restrict__ hist_news,
                 const uint8_t *__restrict__ hist_mask, int32_t max_history, int32_t k, uint64_t *__restrict__ keys_out,
                 int32_t *__restrict__ out_index, float *__restrict__ out_score, int32_t *__restrict__ out_count) {
    extern __shared__ __align__(16) uint64_t smem_keys[];
    uint64_t *buf = smem_keys;           // [slice]  compacted keys of the group
    uint64_t *sel = smem_keys + slice;   // [1024]   the selected keys
    __shared__ int hraw[kHistMax], hsorted[kHistMax];
    __shared__ unsigned bins[256];
    __shared__ int s_nh, s_n, s_nsel, s_bin;
    __shared__ unsigned s_above, s_binc;

    const int tid = threadIdx.x;
    const int64_t u = blockIdx.x / groups;
    const int g = (int)(blockIdx.x - u * groups);
    const int64_t lo = (int64_t)g * slice;
    const int64_t hi = min(n_in, lo + slice);
    if (tid == 0) { s_nh = 0; s_n = 0; s_nsel = 0; }
    __syncthreads();

    const int nh = kScores && hist_news != nullptr ? load_history(hist_news, hist_mask, max_history, u, hraw, hsorted, &s_nh) : 0;

    // ---- load: one read per input, keys compacted into shared memory ----
    for (int64_t i0 = lo; i0 < hi; i0 += kTopkThreads) {
        const int64_t i = i0 + tid;
        bool ok = false;
        uint64_t key = 0;
        if (i < hi) {
            if (kScores) {
                const float s = scores[u * n_in + i];
                ok = returnable(s, i, exclude, pool_news, hsorted, nh);
                if (ok) key = pool_key(s, pool_index[i]);
            } else {
                key = keys_in[u * n_in + i];
                ok = key != 0;
            }
        }
        append_key(ok, key, buf, &s_n, slice);
    }
    __syncthreads();
    const int n = min(s_n, slice);

    // ---- select: the k largest keys of buf[0, n) ----
    const uint64_t *src = buf;
    int cnt = n;
    if (n > k) {
        uint64_t prefix = 0, mask = 0;
        unsigned rem = (unsigned)k;                    // keys still to take below the resolved digits
        for (int shift = 56; shift >= 0; shift -= 8) {
            for (int b = tid; b < 256; b += kTopkThreads) bins[b] = 0;
            __syncthreads();
            for (int i = tid; i < n; i += kTopkThreads) {
                const uint64_t key = buf[i];
                if ((key & mask) == prefix) atomicAdd(&bins[(key >> shift) & 255u], 1u);
            }
            __syncthreads();
            if (tid < 32) {                             // warp 0: the digit holding the rem-th largest matching key
                const int lane = tid;
                unsigned c[8], tot = 0;
#pragma unroll
                for (int j = 0; j < 8; ++j) { c[j] = bins[255 - (lane * 8 + j)]; tot += c[j]; }
                unsigned inc = tot;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const unsigned v = __shfl_up_sync(0xffffffffu, inc, o);
                    if (lane >= o) inc += v;
                }
                unsigned a = inc - tot;
                if (a < rem && rem <= inc) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        if (a + c[j] >= rem) { s_bin = 255 - (lane * 8 + j); s_above = a; s_binc = c[j]; break; }
                        a += c[j];
                    }
                }
            }
            __syncthreads();
            rem -= s_above;
            prefix |= (uint64_t)s_bin << shift;
            mask |= (uint64_t)0xffu << shift;
            const bool whole = s_binc == rem;           // the boundary bin is taken whole: threshold = prefix
            __syncthreads();                            // every thread has read s_* before warp 0 rewrites them
            if (whole) break;
        }
        for (int64_t i0 = 0; i0 < n; i0 += kTopkThreads) {
            const int i = (int)(i0 + tid);
            const uint64_t key = i < n ? buf[i] : 0;
            append_key(i < n && key >= prefix, key, sel, &s_nsel, k);
        }
        __syncthreads();
        src = sel;
        cnt = min(s_nsel, k);
    }

    if (keys_out != nullptr) {
        uint64_t *dst = keys_out + ((int64_t)u * groups + g) * k;
        for (int j = tid; j < k; j += kTopkThreads) dst[j] = j < cnt ? src[j] : 0;
        return;
    }

    // ---- last round: bitonic sort (descending) of the cnt <= k <= 1024 selected keys, then the outputs ----
    int m = 1;
    while (m < cnt) m <<= 1;
    if (src != sel)
        for (int j = tid; j < cnt; j += kTopkThreads) sel[j] = src[j];
    for (int j = cnt + tid; j < m; j += kTopkThreads) sel[j] = 0;
    __syncthreads();
    for (int size = 2; size <= m; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = tid; t < (m >> 1); t += kTopkThreads) {
                const int i = 2 * t - (t & (stride - 1));
                const int j = i + stride;
                const uint64_t a = sel[i], b = sel[j];
                if ((a < b) == ((i & size) == 0)) { sel[i] = b; sel[j] = a; }
            }
            __syncthreads();
        }
    }
    for (int j = tid; j < k; j += kTopkThreads) {
        const bool ok = j < cnt;
        const uint64_t key = ok ? sel[j] : 0;
        out_index[u * k + j] = ok ? (int32_t)~(uint32_t)key : -1;
        out_score[u * k + j] = ok ? ord_score((uint32_t)(key >> 32)) : -INFINITY;
    }
    if (tid == 0) out_count[u] = cnt;
}

// Round plan shared by the scratch query and the launcher: round 0 groups of slice0 scores, later rounds kSliceMax keys.
struct TopkPlan {
    int32_t slice0;
    int64_t groups0, groups1;   // groups of rounds 0 and 1 (1 = that round is the last)
};

static TopkPlan topk_plan(int32_t users, int64_t pool, int32_t k) {
    TopkPlan p;
    const int64_t want = topk_cdiv(2 * (int64_t)num_sms(), users > 0 ? users : 1);    // groups per user for ~2 CTAs / SM
    int64_t s = topk_cdiv(pool, want);
    s = max(s, (int64_t)max(2 * k, 2048));       // >= 2k: every later round folds >= 2 groups into one
    s = min(s, (int64_t)kSliceMax);
    p.slice0 = (int32_t)s;
    p.groups0 = topk_cdiv(pool, s);
    p.groups1 = p.groups0 > 1 ? topk_cdiv(p.groups0 * k, kSliceMax) : 1;
    return p;
}


// ---- ranks of held-out clicks in the whole pool (lime_pool_rank_metrics) ----------------------------------------------
// Count launch: CTA blockIdx.x = u * groups + g over positions [g * slice, (g + 1) * slice) of user u (round 0's groups).
// It builds u's n <= T target keys (eligible, first copy of each position) sorted ascending in shared memory, then
// reads every score of its slice once: an eligible position with key x adds 1 to bin p = #{targets with key < x}
// (p = 0, a position below every target, costs no atomic).  Target j (0-based ascending) then has rank
// 1 + sum_{p > j} bin[p]: the eligible positions above it.  counts[u * (T + 1)] = eligible positions, counts[.. + p] =
// bin p; slot_order[u * T + t] = ascending index of target slot t, -1 = unranked (written by group 0).
constexpr int kRankThreads = kTopkThreads;      // load_history's CTA size
constexpr int kRankMaxT = LIME_POOL_RANK_MAX_TARGETS;
constexpr int kFinishWarps = 4;
constexpr int kMaxColumnsK = 2 + LIME_POOL_RANK_MAX_CUTOFFS;      // nDCG cutoffs 5, 10, then the caller's

struct RankCutoffs {
    int32_t k[LIME_POOL_RANK_MAX_CUTOFFS];
    int32_t n;
};

__global__ void __launch_bounds__(kRankThreads)
pool_rank_count_kernel(const float *__restrict__ scores, int64_t pool, int32_t slice, int32_t groups,
                       const int32_t *__restrict__ pool_index, const int32_t *__restrict__ pool_news,
                       const uint8_t *__restrict__ exclude, const int32_t *__restrict__ hist_news,
                       const uint8_t *__restrict__ hist_mask, int32_t max_history, const int32_t *__restrict__ target_pos,
                       int32_t T, unsigned *__restrict__ counts, int32_t *__restrict__ slot_order) {
    __shared__ int hraw[kHistMax], hsorted[kHistMax];
    __shared__ uint64_t tkey[kRankMaxT], tsorted[kRankMaxT];
    __shared__ int tpos[kRankMaxT];
    __shared__ unsigned bins[kRankMaxT + 1];
    __shared__ int s_nh, s_n;
    __shared__ unsigned s_elig;

    const int tid = threadIdx.x, lane = tid & 31;
    const int64_t u = blockIdx.x / groups;
    const int g = (int)(blockIdx.x - u * groups);
    const int64_t lo = (int64_t)g * slice;
    const int64_t hi = min(pool, lo + slice);
    const float *row = scores + u * pool;
    if (tid == 0) { s_nh = 0; s_n = 0; s_elig = 0; }
    for (int b = tid; b <= T; b += kRankThreads) bins[b] = 0;
    __syncthreads();
    const int nh = hist_news != nullptr ? load_history(hist_news, hist_mask, max_history, u, hraw, hsorted, &s_nh) : 0;

    // ---- targets: key of every eligible slot, later copies of a position dropped, rank-sorted ascending ----
    uint64_t key = 0;
    int pos = -1;
    if (tid < T) {
        pos = target_pos[u * T + tid];
        if (pos >= 0 && pos < pool) {
            const float s = row[pos];
            if (returnable(s, pos, exclude, pool_news, hsorted, nh)) key = pool_key(s, pool_index[pos]);
        }
        if (key == 0) pos = -1;
        tpos[tid] = pos;
    }
    __syncthreads();
    if (key != 0)
        for (int j = 0; j < tid; ++j)
            if (tpos[j] == pos) { key = 0; break; }
    if (tid < T) tkey[tid] = key;
    __syncthreads();
    int r = -1;
    if (key != 0) {
        r = 0;
        for (int j = 0; j < T; ++j) r += tkey[j] != 0 && tkey[j] < key;
        tsorted[r] = key;
        atomicAdd(&s_n, 1);
    }
    if (g == 0 && tid < T) slot_order[u * T + tid] = r;
    __syncthreads();
    const int n = s_n;
    const uint32_t lowest = n > 0 ? (uint32_t)(tsorted[0] >> 32) : 0xffffffffu;

    // ---- positions: eligible count, and bin p of every eligible position above p targets ----
    unsigned elig = 0;
    for (int64_t i0 = lo; i0 < hi; i0 += kRankThreads) {
        const int64_t i = i0 + tid;
        int p = 0;
        if (i < hi) {
            const float s = row[i];
            if (returnable(s, i, exclude, pool_news, hsorted, nh)) {
                ++elig;
                if (n > 0 && score_ord(s) >= lowest) {  // else below every target: p = 0 without reading pool_index
                    const uint64_t x = pool_key(s, pool_index[i]);
                    int a = 0, b = n;                   // p = first slot >= x
                    while (a < b) {
                        const int mid = (a + b) >> 1;
                        if (tsorted[mid] < x) a = mid + 1; else b = mid;
                    }
                    p = a;
                }
            }
        }
        // warp-aggregated increments: a low-ranked target sends most of the pool into one bin
        if (__any_sync(0xffffffffu, p > 0)) {
            const unsigned peers = __match_any_sync(0xffffffffu, p);
            if (p > 0 && lane == __ffs(peers) - 1) atomicAdd(&bins[p], (unsigned)__popc(peers));
        }
    }
    elig = __reduce_add_sync(0xffffffffu, elig);
    if (lane == 0 && elig) atomicAdd(&s_elig, elig);
    __syncthreads();
    unsigned *c = counts + u * (T + 1);
    if (tid == 0 && s_elig) atomicAdd(c, s_elig);
    for (int b = 1 + tid; b <= n; b += kRankThreads)
        if (bins[b]) atomicAdd(c + b, bins[b]);
}


// Finish launch: one warp per user.  Ranks by a suffix sum over the bins (lane l owns bins 8l + 1 .. 8l + 8), written back
// in the caller's slot order; then the counts and the metrics row (lime_rank_metrics' formulas, fp64).
__global__ void __launch_bounds__(kFinishWarps * 32)
pool_rank_finish_kernel(const unsigned *__restrict__ counts, const int32_t *__restrict__ slot_order, int32_t users,
                        int32_t T, RankCutoffs cut, int32_t *__restrict__ out_rank, int32_t *__restrict__ out_ranked,
                        int64_t *__restrict__ out_eligible, double *__restrict__ out_metrics) {
    __shared__ int srank[kFinishWarps][kRankMaxT];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t u = (int64_t)blockIdx.x * kFinishWarps + w;
    if (u >= users) return;
    const unsigned *c = counts + u * (T + 1);
    const int32_t *slot = slot_order + u * T;
    int n = 0;
    for (int t = lane; t < T; t += 32) n += slot[t] >= 0;
    n = __reduce_add_sync(0xffffffffu, n);
    const long long N = c[0];

    constexpr int kPer = kRankMaxT / 32;
    unsigned v[kPer], tot = 0;
#pragma unroll
    for (int m = 0; m < kPer; ++m) {
        const int b = lane * kPer + m + 1;
        v[m] = b <= n ? c[b] : 0u;
        tot += v[m];
    }
    unsigned above = tot;                               // inclusive suffix over lanes >= this one
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned x = __shfl_down_sync(0xffffffffu, above, o);
        if (lane + o < 32) above += x;
    }
    above -= tot;
#pragma unroll
    for (int m = kPer - 1; m >= 0; --m) {              // target j = lane * kPer + m: 1 + bins j + 1 .. n
        above += v[m];
        if (lane * kPer + m < n) srank[w][lane * kPer + m] = 1 + (int)above;
    }
    __syncwarp();
    for (int t = lane; t < T; t += 32) {
        const int o = slot[t];
        out_rank[u * T + t] = o >= 0 ? srank[w][o] : 0;
    }

    const int ncol = 2 + cut.n;
    double *out = out_metrics + u * (4 + 2 * cut.n);
    if (lane == 0) {
        out_ranked[u] = n;
        out_eligible[u] = N;
    }
    if (n == 0) {
        for (int q = lane; q < 4 + 2 * cut.n; q += 32) out[q] = __longlong_as_double(0x7ff8000000000000LL);
        return;
    }
    long long below = 0;                                // sum over targets of N - r
    double rr = 0.0, dcg[kMaxColumnsK], ideal[kMaxColumnsK];
    int hits[kMaxColumnsK];
#pragma unroll
    for (int q = 0; q < kMaxColumnsK; ++q) { dcg[q] = 0.0; ideal[q] = 0.0; hits[q] = 0; }
    for (int j = lane; j < n; j += 32) {
        const int r = srank[w][j];
        below += N - r;
        rr += 1.0 / (double)r;
        const double gr = 1.0 / log2((double)r + 1.0);
        const double gi = 1.0 / log2((double)(j + 1) + 1.0);     // ideal: the ranked targets at 1 .. n
#pragma unroll
        for (int q = 0; q < kMaxColumnsK; ++q) {
            const int K = q == 0 ? 5 : q == 1 ? 10 : (q < ncol ? cut.k[q - 2] : 0);
            if (r <= K) { dcg[q] += gr; hits[q] += 1; }
            if (j + 1 <= K) ideal[q] += gi;
        }
    }
    below = warp_sum_ll(below);
    rr = warp_sum_d(rr);
#pragma unroll
    for (int q = 0; q < kMaxColumnsK; ++q) {
        dcg[q] = warp_sum_d(dcg[q]);
        ideal[q] = warp_sum_d(ideal[q]);
        hits[q] = __reduce_add_sync(0xffffffffu, hits[q]);
    }
    if (lane == 0) {
        const long long nn = n;
        out[0] = (double)(below - nn * (nn - 1) / 2) / ((double)nn * (double)(N - nn));     // NaN when N == n
        out[1] = rr / (double)nn;
        out[2] = dcg[0] / ideal[0];
        out[3] = dcg[1] / ideal[1];
#pragma unroll
        for (int q = 2; q < kMaxColumnsK; ++q)
            if (q < ncol) {
                out[4 + 2 * (q - 2)] = (double)hits[q] / (double)nn;
                out[5 + 2 * (q - 2)] = dcg[q] / ideal[q];
            }
    }
}

}  // namespace lime

using namespace lime;

extern "C" int64_t lime_pool_topk_scratch_bytes(int32_t users, int64_t pool, int32_t k) {
    if (users <= 0 || pool <= 0 || k < 1 || k > LIME_TOPK_MAX) return 0;
    const TopkPlan p = topk_plan(users, pool, k);
    if (p.groups0 == 1) return 0;
    return (int64_t)users * k * (p.groups0 + (p.groups1 > 1 ? p.groups1 : 0)) * (int64_t)sizeof(uint64_t);
}

extern "C" int lime_pool_topk(const float *scores, int32_t users, int64_t pool, const int32_t *pool_index,
                              const int32_t *pool_news, const uint8_t *exclude, const int32_t *hist_news,
                              const uint8_t *hist_mask, int32_t max_history, int32_t k, int32_t *out_index,
                              float *out_score, int32_t *out_count, void *scratch, void *stream) {
    LIME_CHECK_ARG(k >= 1 && k <= LIME_TOPK_MAX, "lime_pool_topk: k=%d not in [1, %d]", k, LIME_TOPK_MAX);
    LIME_CHECK_ARG(scores && pool_index && out_index && out_score && out_count, "lime_pool_topk: null argument");
    LIME_CHECK_ARG(users >= 0, "lime_pool_topk: users=%d < 0", users);
    LIME_CHECK_ARG(pool >= 1 && pool < (1LL << 31), "lime_pool_topk: pool=%lld not in [1, 2^31)", (long long)pool);
    LIME_CHECK_ARG((hist_news == nullptr) == (hist_mask == nullptr), "lime_pool_topk: hist_news and hist_mask go together");
    LIME_CHECK_ARG(hist_news == nullptr || pool_news != nullptr, "lime_pool_topk: the clicked exclusion needs pool_news");
    LIME_CHECK_ARG(hist_news == nullptr || (max_history >= 1 && max_history <= kHistMax),
                   "lime_pool_topk: max_history=%d not in [1, %d]", max_history, kHistMax);
    if (users == 0) return 0;
    const TopkPlan p = topk_plan(users, pool, k);
    LIME_CHECK_ARG((int64_t)users * p.groups0 < (1LL << 31), "lime_pool_topk: users x groups exceeds the grid");
    LIME_CHECK_ARG(p.groups0 == 1 || scratch != nullptr, "lime_pool_topk: null scratch (lime_pool_topk_scratch_bytes = %lld)",
                   (long long)lime_pool_topk_scratch_bytes(users, pool, k));
    cudaStream_t st = as_stream(stream);
    uint64_t *bufA = static_cast<uint64_t *>(scratch);
    uint64_t *bufB = bufA ? bufA + (int64_t)users * k * p.groups0 : nullptr;

    const bool last0 = p.groups0 == 1;
    size_t smem = ((size_t)p.slice0 + LIME_TOPK_MAX) * sizeof(uint64_t);
    LIME_CUDA(cudaFuncSetAttribute(pool_topk_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    pool_topk_kernel<true><<<(unsigned)(users * p.groups0), kTopkThreads, smem, st>>>(
        scores, nullptr, pool, p.slice0, (int32_t)p.groups0, pool_index, pool_news, exclude, hist_news, hist_mask,
        max_history, k, last0 ? nullptr : bufA, out_index, out_score, out_count);
    LIME_LAUNCH_CHECK("pool_topk_kernel<scores>");

    // later rounds: groups x k keys per user -> ceil(groups x k / kSliceMax) groups, ping-pong between the two buffers
    int64_t groups = p.groups0;
    uint64_t *in = bufA, *out = bufB;
    smem = ((size_t)kSliceMax + LIME_TOPK_MAX) * sizeof(uint64_t);
    if (groups > 1) LIME_CUDA(cudaFuncSetAttribute(pool_topk_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    while (groups > 1) {
        const int64_t n_in = groups * k;
        const int64_t next = topk_cdiv(n_in, kSliceMax);
        pool_topk_kernel<false><<<(unsigned)(users * next), kTopkThreads, smem, st>>>(
            nullptr, in, n_in, kSliceMax, (int32_t)next, nullptr, nullptr, nullptr, nullptr, nullptr, 0, k,
            next == 1 ? nullptr : out, out_index, out_score, out_count);
        LIME_LAUNCH_CHECK("pool_topk_kernel<keys>");
        groups = next;
        uint64_t *t = in; in = out; out = t;
    }
    return 0;
}

extern "C" int64_t lime_pool_rank_scratch_bytes(int32_t users, int32_t targets) {
    if (users <= 0 || targets < 1 || targets > LIME_POOL_RANK_MAX_TARGETS) return 0;
    return (int64_t)users * (2 * targets + 1) * (int64_t)sizeof(int32_t);   // counts [users, T + 1], slot_order [users, T]
}

extern "C" int lime_pool_rank_metrics(const float *scores, int32_t users, int64_t pool, const int32_t *pool_index,
                                      const int32_t *pool_news, const uint8_t *exclude, const int32_t *hist_news,
                                      const uint8_t *hist_mask, int32_t max_history, const int32_t *target_pos, int32_t targets,
                                      const int32_t *cutoffs, int32_t num_cutoffs, int32_t *out_rank, int32_t *out_ranked,
                                      int64_t *out_eligible, double *out_metrics, void *scratch, void *stream) {
    LIME_CHECK_ARG(targets >= 1 && targets <= LIME_POOL_RANK_MAX_TARGETS, "lime_pool_rank_metrics: targets=%d not in [1, %d]",
                   targets, LIME_POOL_RANK_MAX_TARGETS);
    LIME_CHECK_ARG(scores && pool_index && target_pos && out_rank && out_ranked && out_eligible && out_metrics && scratch,
                   "lime_pool_rank_metrics: null argument");
    LIME_CHECK_ARG(num_cutoffs >= 0 && num_cutoffs <= LIME_POOL_RANK_MAX_CUTOFFS,
                   "lime_pool_rank_metrics: num_cutoffs=%d not in [0, %d]", num_cutoffs, LIME_POOL_RANK_MAX_CUTOFFS);
    LIME_CHECK_ARG(num_cutoffs == 0 || cutoffs != nullptr, "lime_pool_rank_metrics: null cutoffs");
    RankCutoffs cut = {};
    cut.n = num_cutoffs;
    for (int q = 0; q < num_cutoffs; ++q) {
        LIME_CHECK_ARG(cutoffs[q] >= 1, "lime_pool_rank_metrics: cutoff %d = %d < 1", q, cutoffs[q]);
        cut.k[q] = cutoffs[q];
    }
    LIME_CHECK_ARG(users >= 0, "lime_pool_rank_metrics: users=%d < 0", users);
    LIME_CHECK_ARG(pool >= 1 && pool < (1LL << 31), "lime_pool_rank_metrics: pool=%lld not in [1, 2^31)", (long long)pool);
    LIME_CHECK_ARG((hist_news == nullptr) == (hist_mask == nullptr), "lime_pool_rank_metrics: hist_news and hist_mask go together");
    LIME_CHECK_ARG(hist_news == nullptr || pool_news != nullptr, "lime_pool_rank_metrics: the clicked exclusion needs pool_news");
    LIME_CHECK_ARG(hist_news == nullptr || (max_history >= 1 && max_history <= kHistMax),
                   "lime_pool_rank_metrics: max_history=%d not in [1, %d]", max_history, kHistMax);
    if (users == 0) return 0;
    const TopkPlan p = topk_plan(users, pool, 1);       // round 0's groups: about 2 CTAs per SM even for one user
    LIME_CHECK_ARG((int64_t)users * p.groups0 < (1LL << 31), "lime_pool_rank_metrics: users x groups exceeds the grid");
    cudaStream_t st = as_stream(stream);
    unsigned *counts = static_cast<unsigned *>(scratch);
    int32_t *slot_order = reinterpret_cast<int32_t *>(counts + (int64_t)users * (targets + 1));
    LIME_CUDA(cudaMemsetAsync(counts, 0, (size_t)users * (targets + 1) * sizeof(unsigned), st));
    pool_rank_count_kernel<<<(unsigned)(users * p.groups0), kRankThreads, 0, st>>>(
        scores, pool, p.slice0, (int32_t)p.groups0, pool_index, pool_news, exclude, hist_news, hist_mask, max_history,
        target_pos, targets, counts, slot_order);
    LIME_LAUNCH_CHECK("pool_rank_count_kernel");
    pool_rank_finish_kernel<<<(unsigned)topk_cdiv(users, kFinishWarps), kFinishWarps * 32, 0, st>>>(
        counts, slot_order, users, targets, cut, out_rank, out_ranked, out_eligible, out_metrics);
    LIME_LAUNCH_CHECK("pool_rank_finish_kernel");
    return 0;
}
