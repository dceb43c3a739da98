// Writing freshly built rows into the per-news vector cache (util.build_news_cache / extend_news_cache /
// refresh_news_cache): one pass per row derives every role the scoring kernels read.
#include <cuda_fp16.h>

#include "common.cuh"

namespace lime {
namespace {

constexpr int kRowsPerCta = 8;                        // one warp per row
constexpr int kW = 3 * LIME_D;                        // w1 w2 w3: the columns cand16 splits
constexpr int kHistQ = LIME_HIST_LD / 4;              // float4 per hist row (213)
constexpr int kCandQ = LIME_CAND_LD / 4;              // float4 per cand row (430)
static_assert(LIME_HIST_LD % 4 == 0 && LIME_CAND_LD % 4 == 0 && kW % 8 == 0, "rows must split into 16-byte pieces");
static_assert(LIME_CAND16_LD == 2 * kW, "cand16 row = [hi | lo] of w1 w2 w3");
static_assert(LIME_CAND_ABSMAX == LIME_CAND_SCAL + 7 && LIME_CAND_ABSMAX % 4 == 3, "the absmax column ends a float4");
static_assert(LIME_HIST_TOPIC_ID + 1 == LIME_HIST_GW_ABSMAX && LIME_HIST_TOPIC_ID % 2 == 0, "topic id | gw absmax are one float2");

__device__ __forceinline__ float4 ld4(const float *p) { return *reinterpret_cast<const float4 *>(p); }
__device__ __forceinline__ void st4(float *p, float4 v) { *reinterpret_cast<float4 *>(p) = v; }

// scale * x = hi + lo, the arithmetic of split_f16_pairs_kernel (no contraction of the product into the subtraction)
__device__ __forceinline__ void split_pair(float x, float scale, __half &h, __half &l) {
    const float xs = __fmul_rn(x, scale);
    h = __float2half_rn(xs);
    l = __float2half_rn(__fsub_rn(xs, __half2float(h)));
}

__device__ __forceinline__ float absmax_step(float mx, float x) {
    mx = fmaxf(mx, fabsf(x));
    return x != x ? INFINITY : mx;
}

// One warp per source row r, written at destination row d = dst_rows[r] (rows with d outside [0, news_num) are skipped).
// Plain (coherent) loads: in the in-place form the source row is the destination row.  Every store there writes back the
// value that was read, except the store of cand[1207], whose source value is never used.
__global__ void __launch_bounds__(32 * kRowsPerCta) cache_write_rows_kernel(
    const float *hist, const float *cand, int64_t n, const int64_t *__restrict__ dst_rows, float *hist_rows, float *cand_rows,
    __half *__restrict__ cand16, float *__restrict__ news_meta, float *__restrict__ hist_vg, int64_t news_num, float scale) {
    const int lane = threadIdx.x & 31;
    const int64_t r = (int64_t)blockIdx.x * kRowsPerCta + (threadIdx.x >> 5);
    if (r >= n) return;
    const int64_t d = dst_rows[r];
    if (d < 0 || d >= news_num) return;
    const float *hs = hist + r * LIME_HIST_LD, *cs = cand + r * LIME_CAND_LD;
    float *hd = hist_rows + d * LIME_HIST_LD, *cd = cand_rows + d * LIME_CAND_LD;

    // w1 w2 w3: copy, fp16 hi / lo pair, max |w|; 8 columns per step -> one 16-byte store per image
    __half *c16 = cand16 + d * LIME_CAND16_LD;
    float mx = 0.0f;
    for (int e = lane * 8; e < kW; e += 32 * 8) {
        const float4 a = ld4(cs + e), b = ld4(cs + e + 4);
        st4(cd + e, a);
        st4(cd + e + 4, b);
        const float x[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        __align__(16) __half hi[8], lo[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            split_pair(x[i], scale, hi[i], lo[i]);
            mx = absmax_step(mx, x[i]);
        }
        *reinterpret_cast<uint4 *>(c16 + e) = *reinterpret_cast<const uint4 *>(hi);
        *reinterpret_cast<uint4 *>(c16 + kW + e) = *reinterpret_cast<const uint4 *>(lo);
    }
    mx = warp_max(mx);

    // the rest of the cand row, max |w| stamped into LIME_CAND_ABSMAX
    for (int q = kW / 4 + lane; q < kCandQ; q += 32) {
        float4 v = ld4(cs + 4 * q);
        if (4 * q + 3 == LIME_CAND_ABSMAX) v.w = mx;
        st4(cd + 4 * q, v);
    }
    // hist row; vc and gw also interleaved by 4 dims into hist_vg (v0..3 g0..3 v4..7 ...)
    float *vg = hist_vg + d * 2 * LIME_D;
    for (int q = lane; q < LIME_D / 4; q += 32) {
        const float4 v = ld4(hs + LIME_HIST_VC + 4 * q), g = ld4(hs + LIME_HIST_GW + 4 * q);
        st4(hd + LIME_HIST_VC + 4 * q, v);
        st4(hd + LIME_HIST_GW + 4 * q, g);
        st4(vg + 8 * q, v);
        st4(vg + 8 * q + 4, g);
    }
    for (int q = LIME_HIST_T / 4 + lane; q < kHistQ; q += 32) st4(hd + 4 * q, ld4(hs + 4 * q));
    // news_meta sector: topic id | gw absmax | w absmax | B1 B2 B3 cb | 0
    if (lane == 0) {
        const float2 t = *reinterpret_cast<const float2 *>(hs + LIME_HIST_TOPIC_ID);
        const float4 s = ld4(cs + LIME_CAND_SCAL);            // columns 1200..1203
        const float4 u = ld4(cs + LIME_CAND_SCAL + 4);        // 1204..1207 (1207 is the stale absmax: not used)
        float *m = news_meta + d * LIME_META_LD;
        st4(m, make_float4(t.x, t.y, mx, s.w));
        st4(m + 4, make_float4(u.x, u.y, u.z, 0.0f));
    }
}

}  // namespace
}  // namespace lime

extern "C" int lime_cache_write_rows(const float *hist, const float *cand, int64_t n, const int64_t *dst_rows, float *hist_rows,
                                     float *cand_rows, void *cand16, float *news_meta, float *hist_vg, int64_t news_num,
                                     void *stream) {
    LIME_CHECK_ARG(hist && cand && dst_rows && hist_rows && cand_rows && cand16 && news_meta && hist_vg,
                   "lime_cache_write_rows: null argument");
    LIME_CHECK_ARG(n >= 0 && news_num >= 1 && news_num <= INT32_MAX, "lime_cache_write_rows: n=%lld news_num=%lld", (long long)n,
                   (long long)news_num);
    const uintptr_t any = (uintptr_t)hist | (uintptr_t)cand | (uintptr_t)hist_rows | (uintptr_t)cand_rows | (uintptr_t)cand16 |
                          (uintptr_t)news_meta | (uintptr_t)hist_vg;
    LIME_CHECK_ARG((any & 15) == 0 && ((uintptr_t)dst_rows & 7) == 0, "lime_cache_write_rows: arrays must be 16-byte aligned");
    if (n == 0) return 0;
    const int64_t grid = (n + lime::kRowsPerCta - 1) / lime::kRowsPerCta;
    LIME_CHECK_ARG(grid <= INT32_MAX, "lime_cache_write_rows: n=%lld too large", (long long)n);
    lime::cache_write_rows_kernel<<<(unsigned)grid, 32 * lime::kRowsPerCta, 0, lime::as_stream(stream)>>>(
        hist, cand, n, dst_rows, hist_rows, cand_rows, reinterpret_cast<__half *>(cand16), news_meta, hist_vg, news_num,
        LIME_CAND16_SCALE);
    LIME_LAUNCH_CHECK("cache_write_rows_kernel");
    return 0;
}
