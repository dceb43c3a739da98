// Ranking + AUC / MRR / nDCG@5 / nDCG@10 per impression (sm_100a).
//
// Replaces compute_scores' tail (util.py:113-123: group by impression, stable sort by score
// descending, rank = 1-based position) and evaluate.scoring's per-impression body
// (evaluate.py:64-80) with y_score = 1/rank.  Ranks are distinct, so sklearn's roc_auc_score is the
// fraction of (positive, negative) pairs with the positive ranked first; counted in integers.
// The reference does all of this in Python through two text files; here one warp owns an
// impression and everything stays on the device.
#include "common.cuh"

namespace lime {

constexpr int kMetricWarps = 4;

__global__ void __launch_bounds__(kMetricWarps * 32)
rank_metrics_kernel(const float *__restrict__ scores, const uint8_t *__restrict__ labels,
                    const int64_t *__restrict__ cand_off, int64_t num_impressions,
                    int32_t *__restrict__ ranks, double *__restrict__ metrics) {
    const int lane = threadIdx.x & 31;
    const int64_t imp = (int64_t)blockIdx.x * kMetricWarps + (threadIdx.x >> 5);
    if (imp >= num_impressions) return;
    const int64_t p0 = cand_off[imp];
    const int n = (int)(cand_off[imp + 1] - p0);
    double *out = metrics + imp * 4;
    if (n <= 0) {   // masked impression: skipped by the mean (evaluate.py:44-45)
        if (lane < 4) out[lane] = __longlong_as_double(0x7ff8000000000000LL);
        return;
    }
    const float *s = scores + p0;
    const uint8_t *y = labels + p0;
    long long npos = 0, pos_below = 0;   // pos_below = sum over positives of (n - rank)
    double rr = 0.0, dcg5 = 0.0, dcg10 = 0.0;
    for (int j = lane; j < n; j += 32) {
        const float sj = s[j];
        int rank = 1;
        for (int k = 0; k < n; ++k) {
            const float sk = s[k];
            rank += (sk > sj) || (sk == sj && k < j);   // stable: earlier candidate wins a tie
        }
        if (ranks) ranks[p0 + j] = rank;
        if (y[j]) {
            npos += 1;
            pos_below += n - rank;
            rr += 1.0 / (double)rank;
            const double g = 1.0 / log2((double)rank + 1.0);
            if (rank <= 5) dcg5 += g;
            if (rank <= 10) dcg10 += g;
        }
    }
    npos = warp_sum_ll(npos);
    pos_below = warp_sum_ll(pos_below);
    rr = warp_sum_d(rr);
    dcg5 = warp_sum_d(dcg5);
    dcg10 = warp_sum_d(dcg10);
    if (lane == 0) {
        const long long nneg = n - npos;
        double ideal5 = 0.0, ideal10 = 0.0;
        for (int i = 1; i <= 10 && i <= npos; ++i) {
            const double g = 1.0 / log2((double)i + 1.0);
            if (i <= 5) ideal5 += g;
            ideal10 += g;
        }
        const long long concordant = pos_below - npos * (npos - 1) / 2;
        out[0] = (double)concordant / ((double)npos * (double)nneg);   // NaN when single-class, like the reference's failure
        out[1] = rr / (double)npos;
        out[2] = dcg5 / ideal5;
        out[3] = dcg10 / ideal10;
    }
}

// Deterministic fixed-order sum: one block, each thread a strided fp64 partial, then a tree.
__global__ void __launch_bounds__(1024)
metrics_reduce_kernel(const double *__restrict__ metrics, int64_t n, double *__restrict__ sums) {
    __shared__ double sh[5][1024];
    double acc[5] = {0, 0, 0, 0, 0};
    for (int64_t i = threadIdx.x; i < n; i += 1024) {
        const double a = metrics[i * 4];
        if (a == a || metrics[i * 4 + 1] == metrics[i * 4 + 1]) {   // not the all-NaN "skipped" row
            acc[0] += a;
            acc[1] += metrics[i * 4 + 1];
            acc[2] += metrics[i * 4 + 2];
            acc[3] += metrics[i * 4 + 3];
            acc[4] += 1.0;
        }
    }
    for (int q = 0; q < 5; ++q) sh[q][threadIdx.x] = acc[q];
    __syncthreads();
    for (int w = 512; w > 0; w >>= 1) {
        if (threadIdx.x < w)
            for (int q = 0; q < 5; ++q) sh[q][threadIdx.x] += sh[q][threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x < 5) sums[threadIdx.x] = sh[threadIdx.x][0];
}

}  // namespace lime

using namespace lime;

extern "C" int lime_rank_metrics(const float *scores, const uint8_t *labels, const int64_t *cand_off,
                                 int64_t num_impressions, int32_t *ranks, double *metrics,
                                 void *stream) {
    LIME_CHECK_ARG(scores && labels && cand_off && metrics, "lime_rank_metrics: null argument");
    if (num_impressions <= 0) return 0;
    const int64_t blocks = (num_impressions + kMetricWarps - 1) / kMetricWarps;
    LIME_CHECK_ARG(blocks < (1LL << 31), "lime_rank_metrics: too many impressions");
    rank_metrics_kernel<<<(unsigned)blocks, kMetricWarps * 32, 0, as_stream(stream)>>>(
        scores, labels, cand_off, num_impressions, ranks, metrics);
    LIME_LAUNCH_CHECK("rank_metrics_kernel");
    return 0;
}

extern "C" int lime_metrics_reduce(const double *metrics, int64_t num_impressions, double *sums,
                                   void *stream) {
    LIME_CHECK_ARG(metrics && sums, "lime_metrics_reduce: null argument");
    metrics_reduce_kernel<<<1, 1024, 0, as_stream(stream)>>>(metrics, num_impressions, sums);
    LIME_LAUNCH_CHECK("metrics_reduce_kernel");
    return 0;
}
