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

    int nh = 0;
    if (kScores && hist_news != nullptr) {
        for (int h0 = 0; h0 < max_history; h0 += kTopkThreads) {     // masked-in ids of the history, then rank-sorted
            const int h = h0 + tid;
            const bool ok = h < max_history && hist_mask[u * max_history + h] != 0;
            const unsigned m = __ballot_sync(0xffffffffu, ok);
            if (m) {
                const int lane = tid & 31, leader = __ffs(m) - 1;
                int base = 0;
                if (lane == leader) base = atomicAdd(&s_nh, __popc(m));
                base = __shfl_sync(0xffffffffu, base, leader);
                if (ok) hraw[base + __popc(m & ((1u << lane) - 1u))] = hist_news[u * max_history + h];
            }
        }
        __syncthreads();
        nh = s_nh;
        for (int t = tid; t < nh; t += kTopkThreads) {
            const int v = hraw[t];
            int r = 0;
            for (int j = 0; j < nh; ++j) r += hraw[j] < v || (hraw[j] == v && j < t);
            hsorted[r] = v;
        }
        __syncthreads();
    }

    // ---- load: one read per input, keys compacted into shared memory ----
    for (int64_t i0 = lo; i0 < hi; i0 += kTopkThreads) {
        const int64_t i = i0 + tid;
        bool ok = false;
        uint64_t key = 0;
        if (i < hi) {
            if (kScores) {
                const float s = scores[u * n_in + i];
                ok = s == s && !(exclude != nullptr && exclude[i]);
                if (ok && nh > 0) {
                    const int nw = pool_news[i];
                    int a = 0, b = nh;                    // first slot >= nw
                    while (a < b) {
                        const int mid = (a + b) >> 1;
                        if (hsorted[mid] < nw) a = mid + 1; else b = mid;
                    }
                    ok = !(a < nh && hsorted[a] == nw);
                }
                if (ok) key = ((uint64_t)score_ord(s) << 32) | (uint32_t)~(uint32_t)pool_index[i];
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
