// Stage B: impression scoring on cached news vectors (sm_100a).
//
// One kernel replaces, per (user, candidate) pair, the reference's
//   CandidateAware_ClickedNewsAttention.forward   layers.py:52-93
//   userEncoders.CROWN.forward tail               userEncoders.py:121,151-171
//   RemainingLifetimeWeighting.forward            util.py:23-49
// for the eval layout (one candidate per sample, model.py:158-169).
//
// Algebra (DESIGN.md §"Scoring kernel"): with v_h the cached LIME vector of history slot h,
//   a      = softmax_h( sum_heads softmax_h( Q_head . K_{h,head} / 20, masked ) )      [phase 1]
//   o_h    = v_h * (e + a_h) / (e + 1),  e = exp(-(a_h * (W_g v_h) + b_g))            [phase 2]
//            (== gate*a_h*v_h + (1-gate)*v_h with gate = sigmoid(W_g (a_h v_h) + b_g))
//   x_h    = LayerNorm(o_h)
//   g_h    = W_l m + b_l + W_r x_h,   m = mean of the first P rows of [x ; user_node_embedding]
//   alpha  = softmax_h( (W_K g_h) . (W_Q c + b_Q) / 20 ) = softmax_h( x_h . p / 20 ),  p = (W_K W_r)^T (W_Q c + b_Q)
//   score  = ( m . (W_l^T c) + b_l . c + sum_h alpha_h x_h . (W_r^T c) ) * w(remaining lifetime)
// so a pair needs, per history row, five reductions over the 400 dims
//   S0 = sum o, S1 = sum o^2, D1 = sum o*(gamma*p/20), D2 = sum o*(gamma*W_r^T c), D3 = sum o*(gamma*W_l^T c)
// (the LayerNorm is folded into the dots).  Everything linear in c is cached per news / per
// lifetime-bucket pair at cache-build time (cand_rows / cand_tab).
//
// Thread mapping (phase 2, the hot loop): 16 warps; a warp owns 3-4 history rows; a lane holds dims
// d = lane + 32*j (j < 13) of W_g v_h in REGISTERS (v_h in warp-private shared rows), so the
// per-candidate loop touches only shared memory: one conflict-free LDS.128 fetches
// (gate bias, w1, w2, w3)[d] and is reused by the 4 rows (0.25 LDS per element).  The 4x5 partial
// sums of a warp are reduced with a split butterfly (30 shuffles instead of 100).
// A work unit is <= tile_c consecutive candidates of one impression; CTAs are persistent (one per
// SM) and pull units from a global counter.
#include <type_traits>

#include "common.cuh"
#include "score_common.cuh"

namespace lime {

constexpr int kD = LIME_D;
constexpr int kEPL = kD / 8;        // elements per lane (50)
constexpr int kWarps = 16;                  // 4 per SM sub-partition: balanced issue, 128 registers/thread
constexpr int kThreads = kWarps * 32;
constexpr int kRowsPerWarp = 4;
constexpr int kRowsPerChunk = kWarps * kRowsPerWarp;   // up to 64 history rows resident per pass
constexpr int kSlots = (kD + 31) / 32;      // 13 register slots per lane and row (d = lane + 32 j)
constexpr int kTStride = LIME_TOPIC + 1;    // 51: conflict-free column reads of the topic tile
constexpr int kTqStride = 12;               // heads padded 10 -> 12 (3 x LDS.128)
constexpr int kTqWarp = LIME_TOPIC * kTqStride + kTqStride;   // 612 floats per warp
constexpr int kNW = 3 * kD;                 // 1200 candidate-vector floats staged per candidate

// Phase-2 dim mapping: lane owns dims 128*jp + 4*lane + e (jp < 3, e < 4; register slot 4*jp + e) and,
// for lane < 16, dim 384 + lane (slot 12).  v rows keep the natural order (one LDS.128 per jp); the
// candidate float4s are stored at wpos(d) so that slot s of all lanes is one contiguous 512-byte row.
__device__ __forceinline__ int wpos(int d) {
    return d < 384 ? ((((d >> 7) << 2) + (d & 3)) << 5) + ((d & 127) >> 2) : d;
}

__device__ __forceinline__ void accum5(float (&acc)[5], float o, const float4 &q) {
    acc[0] += o;
    acc[1] = fmaf(o, o, acc[1]);
    acc[2] = fmaf(o, q.y, acc[2]);
    acc[3] = fmaf(o, q.z, acc[3]);
    acc[4] = fmaf(o, q.w, acc[4]);
}

struct SmemLayout {
    float4 *wbuf;      // [2][kD]   (gate bias', w1, w2, w3) per dim, double buffered
    float *v_s;        // [kRowsPerChunk][kD] LIME vectors of the chunk's history rows (warp-private rows)
    float *t_s;        // [H][kTStride]  topic representation of the history slots
    float *a_s;        // [tile_c][H]    candidate-aware attention weights
    float *lg_s;       // [tile_c][H]    x_h . p / 20
    float *y_s;        // [tile_c][H]    x_h . W_r^T c
    float *z_s;        // [tile_c][H]    x_h . W_l^T c
    float *tq_s;       // [kWarps][kTqWarp]
    float *cscal;      // [tile_c][8]    W1s W2s W3s B1 B2 B3 cb  (news part + table part)
    float *cw;         // [tile_c]       lifetime weight
    int *cnews;        // [tile_c]
    int *ctab;         // [tile_c]
    int *cP;           // [tile_c]
    int *hnews;        // [H]
    int *htab;         // [H]
    int *hmask;        // [H]
    int *unit_bcast;   // [4]
};

__host__ __device__ inline size_t align16(size_t x) { return (x + 15) & ~size_t(15); }

__host__ __device__ inline size_t smem_carve(SmemLayout *L, unsigned char *base, int H, int TC) {
    size_t off = 0;
    auto take = [&](size_t bytes) {
        size_t o = off;
        off = align16(off + bytes);
        return o;
    };
    size_t o_wbuf = take(sizeof(float4) * 2 * kD);
    size_t o_v = take(sizeof(float) * kRowsPerChunk * kD);
    size_t o_t = take(sizeof(float) * H * kTStride);
    size_t o_a = take(sizeof(float) * TC * H);
    size_t o_lg = take(sizeof(float) * TC * H);
    size_t o_y = take(sizeof(float) * TC * H);
    size_t o_z = take(sizeof(float) * TC * H);
    size_t o_tq = take(sizeof(float) * kWarps * kTqWarp);
    size_t o_cs = take(sizeof(float) * TC * 8);
    size_t o_cw = take(sizeof(float) * TC);
    size_t o_cn = take(sizeof(int) * TC);
    size_t o_ct = take(sizeof(int) * TC);
    size_t o_cp = take(sizeof(int) * TC);
    size_t o_hn = take(sizeof(int) * H);
    size_t o_ht = take(sizeof(int) * H);
    size_t o_hm = take(sizeof(int) * H);
    size_t o_ub = take(sizeof(int) * 4);
    if (L) {
        L->wbuf = reinterpret_cast<float4 *>(base + o_wbuf);
        L->v_s = reinterpret_cast<float *>(base + o_v);
        L->t_s = reinterpret_cast<float *>(base + o_t);
        L->a_s = reinterpret_cast<float *>(base + o_a);
        L->lg_s = reinterpret_cast<float *>(base + o_lg);
        L->y_s = reinterpret_cast<float *>(base + o_y);
        L->z_s = reinterpret_cast<float *>(base + o_z);
        L->tq_s = reinterpret_cast<float *>(base + o_tq);
        L->cscal = reinterpret_cast<float *>(base + o_cs);
        L->cw = reinterpret_cast<float *>(base + o_cw);
        L->cnews = reinterpret_cast<int *>(base + o_cn);
        L->ctab = reinterpret_cast<int *>(base + o_ct);
        L->cP = reinterpret_cast<int *>(base + o_cp);
        L->hnews = reinterpret_cast<int *>(base + o_hn);
        L->htab = reinterpret_cast<int *>(base + o_ht);
        L->hmask = reinterpret_cast<int *>(base + o_hm);
        L->unit_bcast = reinterpret_cast<int *>(base + o_ub);
    }
    return off;
}

// Per-pair terms of the score for lime_explain_pairs: [pair][H] rows for alpha / topic_attn / contrib, [pair] for
// bias / weight.  Unused (all NULL) by the scoring instantiations.
struct ExplainOut {
    float *alpha;
    float *topic_attn;
    float *contrib;
    float *bias;
    float *weight;
};

// kExplain: phase 3 also writes the decomposition score = bias + sum_h contrib[h] (lime_explain_pairs); the score
// itself is the same expression in both instantiations.
template <int MAXP, bool kExplain>
__global__ void __launch_bounds__(kThreads, 1) score_kernel(const ScoreArgs args, const ExplainOut ex) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const LimeNewsCache &C = args.cache;
    const LimeImpressions &I = args.imp;
    const int H = I.max_history;
    const int TC = I.tile_c;
    SmemLayout S;
    smem_carve(&S, smem_raw, H, TC);

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;
    const int nb = C.num_buckets;
    const int passes = (H + 31) >> 5;
    const int chunks = (H + kRowsPerChunk - 1) / kRowsPerChunk;

    // gate bias' = -log2(e) * b_g lives in .x of both staging buffers for the kernel's lifetime
    for (int d = tid; d < 2 * kD; d += kThreads) S.wbuf[(d / kD) * kD + wpos(d % kD)].x = C.gate_bias[d % kD];

    for (;;) {
        __syncthreads();   // previous unit fully consumed (also orders the .x init above)
        if (tid == 0) S.unit_bcast[0] = atomicAdd(args.work_counter, 1);
        __syncthreads();
        int unit = S.unit_bcast[0];
        if (args.unit_list != nullptr) {
            if (unit >= *args.unit_list_count) break;
            unit = args.unit_list[unit];
        } else if (unit >= I.num_units) {
            break;
        }
        const int imp = I.unit_imp[unit];
        const int pair0 = I.unit_pair0[unit];
        const int cnt = I.unit_count[unit];
        if constexpr (kExplain) {
            if (cnt <= 0) continue;   // a user whose explained news are all padding
        }

        // ---------------- phase 0: unit metadata + topic tile -----------------------------------
        for (int h = tid; h < H; h += kThreads) {
            const long long o = (long long)imp * H + h;
            int n = I.hist_news[o];
            n = (n < 0 || n >= C.news_num) ? 0 : n;
            S.hnews[h] = n;
            S.hmask[h] = I.hist_mask[o];
            const int bf = bucketize_seconds(I.hist_fresh[o], args.bucket_scale, nb);
            const int bl = bucketize_seconds(I.hist_life[o], args.bucket_scale, nb);
            S.htab[h] = bf * nb + bl;
        }
        for (int c = tid; c < cnt; c += kThreads) {
            const long long p = (long long)pair0 + c;
            int n = I.cand_news[p];
            n = (n < 0 || n >= C.news_num) ? 0 : n;
            S.cnews[c] = n;
            const float fr = I.cand_fresh[p], lf = I.cand_life[p];
            S.ctab[c] = bucketize_seconds(fr, args.bucket_scale, nb) * nb +
                        bucketize_seconds(lf, args.bucket_scale, nb);
            S.cw[c] = lifetime_weight(I.cand_remaining ? I.cand_remaining[p] : __fsub_rn(lf, fr), C);
            S.cP[c] = (args.pair_index_base + p >= args.tail_start) ? args.prefix_tail : args.prefix_main;
        }
        __syncthreads();
        for (int idx = tid; idx < H * LIME_TOPIC; idx += kThreads) {
            const int h = idx / LIME_TOPIC, k = idx - h * LIME_TOPIC;
            S.t_s[h * kTStride + k] = C.hist_rows[(size_t)S.hnews[h] * LIME_HIST_LD + LIME_HIST_T + k];
        }
        __syncthreads();

        // ---------------- phase 1: candidate-aware attention weights a[c][h] ---------------------
        // layers.py:66-81 with N = 1 (query weight softmax over a single candidate == 1).
        for (int c = warp; c < cnt; c += kWarps) {
            float *tq = S.tq_s + warp * kTqWarp;
            const float *crow = C.cand_rows + (size_t)S.cnews[c] * LIME_CAND_LD;
            for (int idx = lane; idx < LIME_TOPIC * LIME_CA_HEADS; idx += 32) {
                const int k = idx / LIME_CA_HEADS, hd = idx - k * LIME_CA_HEADS;
                tq[k * kTqStride + hd] = crow[LIME_CAND_TQ + idx];
            }
            if (lane < LIME_CA_HEADS) tq[LIME_TOPIC * kTqStride + lane] = crow[LIME_CAND_QB + lane];
            if (lane < 8) {
                const float tabv = C.cand_tab[(size_t)S.ctab[c] * LIME_CTAB_LD + LIME_CAND_SCAL + lane];
                S.cscal[c * 8 + lane] = crow[LIME_CAND_SCAL + lane] + tabv;
            }
            __syncwarp();

            float sc[MAXP][LIME_CA_HEADS];
#pragma unroll
            for (int p = 0; p < MAXP; ++p) {
                if (p < passes) {
                    const int hh = lane + 32 * p;
                    const bool valid = hh < H;
                    const float *trow = S.t_s + (valid ? hh : 0) * kTStride;
                    float acc[LIME_CA_HEADS];
#pragma unroll
                    for (int hd = 0; hd < LIME_CA_HEADS; ++hd) acc[hd] = tq[LIME_TOPIC * kTqStride + hd];
#pragma unroll 5
                    for (int k = 0; k < LIME_TOPIC; ++k) {
                        const float tv = trow[k];
                        const float4 q0 = *reinterpret_cast<const float4 *>(tq + k * kTqStride);
                        const float4 q1 = *reinterpret_cast<const float4 *>(tq + k * kTqStride + 4);
                        const float2 q2 = *reinterpret_cast<const float2 *>(tq + k * kTqStride + 8);
                        acc[0] = fmaf(q0.x, tv, acc[0]);
                        acc[1] = fmaf(q0.y, tv, acc[1]);
                        acc[2] = fmaf(q0.z, tv, acc[2]);
                        acc[3] = fmaf(q0.w, tv, acc[3]);
                        acc[4] = fmaf(q1.x, tv, acc[4]);
                        acc[5] = fmaf(q1.y, tv, acc[5]);
                        acc[6] = fmaf(q1.z, tv, acc[6]);
                        acc[7] = fmaf(q1.w, tv, acc[7]);
                        acc[8] = fmaf(q2.x, tv, acc[8]);
                        acc[9] = fmaf(q2.y, tv, acc[9]);
                    }
                    const bool keep = valid && (S.hmask[valid ? hh : 0] != 0);
#pragma unroll
                    for (int hd = 0; hd < LIME_CA_HEADS; ++hd)
                        sc[p][hd] = valid ? (keep ? acc[hd] : -1e9f) : -INFINITY;   // masked_fill(mask==0,-1e9)
                } else {
#pragma unroll
                    for (int hd = 0; hd < LIME_CA_HEADS; ++hd) sc[p][hd] = -INFINITY;
                }
            }
            float agg[MAXP];
#pragma unroll
            for (int p = 0; p < MAXP; ++p) agg[p] = 0.0f;
#pragma unroll
            for (int hd = 0; hd < LIME_CA_HEADS; ++hd) {
                float m = -INFINITY;
#pragma unroll
                for (int p = 0; p < MAXP; ++p) m = fmaxf(m, sc[p][hd]);
                m = warp_max(m);
                float e[MAXP];
                float l = 0.0f;
#pragma unroll
                for (int p = 0; p < MAXP; ++p) {
                    e[p] = __expf(sc[p][hd] - m);   // -inf rows (h >= H) give 0
                    l += e[p];
                }
                l = warp_sum(l);
                const float inv = __fdividef(1.0f, l);
#pragma unroll
                for (int p = 0; p < MAXP; ++p) agg[p] = fmaf(e[p], inv, agg[p]);
            }
            // second, unmasked softmax over the history (layers.py:81)
            float m2 = -INFINITY;
#pragma unroll
            for (int p = 0; p < MAXP; ++p) {
                const bool valid = (p < passes) && (lane + 32 * p < H);
                m2 = fmaxf(m2, valid ? agg[p] : -INFINITY);
            }
            m2 = warp_max(m2);
            float l2 = 0.0f;
#pragma unroll
            for (int p = 0; p < MAXP; ++p) {
                const bool valid = (p < passes) && (lane + 32 * p < H);
                agg[p] = valid ? __expf(agg[p] - m2) : 0.0f;
                l2 += agg[p];
            }
            l2 = warp_sum(l2);
            const float inv2 = __fdividef(1.0f, l2);
#pragma unroll
            for (int p = 0; p < MAXP; ++p) {
                const int hh = lane + 32 * p;
                if (p < passes && hh < H) S.a_s[c * H + hh] = agg[p] * inv2;
            }
            __syncwarp();
        }
        __syncthreads();

        // ---------------- phase 2: gated residual + LayerNorm statistics + 3 dots per row --------
        for (int chunk = 0; chunk < chunks; ++chunk) {
            // balanced split of the chunk's rows over the 16 warps (H = 50: two warps take 4 rows, the
            // others 3); the extra rows go to the highest warp ids, which the issue arbiter favours
            const int R = min(kRowsPerChunk, H - chunk * kRowsPerChunk);
            const int rbase = R / kWarps, rrem = R % kWarps;
            const int wfirst = kWarps - rrem;                 // warps >= wfirst own rbase + 1 rows
            const int nrows = rbase + (warp >= wfirst ? 1 : 0);
            const int h0 = chunk * kRowsPerChunk + warp * rbase + max(warp - wfirst, 0);
            // W_g v lives in registers, v itself in this warp's private rows of the shared v tile (16
            // warps = 4 per SM sub-partition caps a thread at 128 registers)
            float gw[kRowsPerWarp][kSlots];
            float *vrow = S.v_s + (size_t)warp * kRowsPerWarp * kD;
#pragma unroll
            for (int r = 0; r < kRowsPerWarp; ++r) {
                const bool row_ok = r < nrows;
                const int hn = row_ok ? S.hnews[h0 + r] : 0;
                const int ht = row_ok ? S.htab[h0 + r] : 0;
                const float *hr = C.hist_rows + (size_t)hn * LIME_HIST_LD;
                const float *tr = C.hist_tab + (size_t)ht * LIME_HTAB_LD;
#pragma unroll
                for (int jp = 0; jp < 3; ++jp) {
                    const int d = 128 * jp + 4 * lane;
                    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
                    const float4 v1 = row_ok ? *reinterpret_cast<const float4 *>(hr + LIME_HIST_VC + d) : z4;
                    const float4 v2 = row_ok ? *reinterpret_cast<const float4 *>(tr + d) : z4;
                    const float4 g1 = row_ok ? *reinterpret_cast<const float4 *>(hr + LIME_HIST_GW + d) : z4;
                    const float4 g2 = row_ok ? *reinterpret_cast<const float4 *>(tr + kD + d) : z4;
                    *reinterpret_cast<float4 *>(vrow + r * kD + d) =
                        make_float4(v1.x + v2.x, v1.y + v2.y, v1.z + v2.z, v1.w + v2.w);
                    gw[r][4 * jp + 0] = g1.x + g2.x;
                    gw[r][4 * jp + 1] = g1.y + g2.y;
                    gw[r][4 * jp + 2] = g1.z + g2.z;
                    gw[r][4 * jp + 3] = g1.w + g2.w;
                }
                const bool tail = row_ok && lane < 16;
                if (lane < 16) vrow[r * kD + 384 + lane] = tail ? (hr[LIME_HIST_VC + 384 + lane] + tr[384 + lane]) : 0.0f;
                gw[r][12] = tail ? (hr[LIME_HIST_GW + 384 + lane] + tr[kD + 384 + lane]) : 0.0f;
            }
            __syncwarp();
            // stage candidate 0
            for (int idx = tid; idx < kNW; idx += kThreads) {
                const int which = idx / kD, d = idx - which * kD;
                const float val = C.cand_rows[(size_t)S.cnews[0] * LIME_CAND_LD + idx] +
                                  C.cand_tab[(size_t)S.ctab[0] * LIME_CTAB_LD + idx];
                reinterpret_cast<float *>(S.wbuf + wpos(d))[1 + which] = val;
            }
            __syncthreads();
            for (int c = 0; c < cnt; ++c) {
                const int buf = c & 1;
                // prefetch the next candidate's folded vectors (news part, bucket-table part); the add
                // and the shared-memory store happen after this candidate's math so the loads overlap it
                float nvr[3], nvt[3];
                const bool has_next = (c + 1 < cnt);
                if (has_next) {
                    const float *cr = C.cand_rows + (size_t)S.cnews[c + 1] * LIME_CAND_LD;
                    const float *ct = C.cand_tab + (size_t)S.ctab[c + 1] * LIME_CTAB_LD;
#pragma unroll
                    for (int q = 0; q < 3; ++q) {
                        const int idx = tid + q * kThreads;
                        nvr[q] = (idx < kNW) ? cr[idx] : 0.0f;
                        nvt[q] = (idx < kNW) ? ct[idx] : 0.0f;
                    }
                }
                const float4 *wb = S.wbuf + buf * kD + lane;
                const float *ac = S.a_s + c * H + h0;
                float k1[5];
                // compile-time row count: one warp-uniform branch per candidate instead of one per element
                auto rows = [&](auto nr_tag) {
                    constexpr int NR = decltype(nr_tag)::value;
                    float a[NR], oma[NR], acc[kRowsPerWarp][5];
#pragma unroll
                    for (int r = 0; r < kRowsPerWarp; ++r)
#pragma unroll
                        for (int q = 0; q < 5; ++q) acc[r][q] = 0.0f;
#pragma unroll
                    for (int r = 0; r < NR; ++r) {
                        a[r] = ac[r];
                        oma[r] = 1.0f - a[r];
                    }
                    // o = v (1 - (1 - a) sigmoid(a W_g v + b_g)), sigmoid(z) = 1 / (1 + 2^z'), z' = -log2(e) z.
                    // Two elements share one MUFU.RCP: 1/x = y / (x y).  z' is clamped to 60 so the product of
                    // two denominators stays finite (gate <= 2^-60 there, i.e. 0 in fp32 arithmetic).
#pragma unroll
                    for (int jp = 0; jp < 3; ++jp) {
                        float4 v4[NR];
#pragma unroll
                        for (int r = 0; r < NR; ++r)
                            v4[r] = *reinterpret_cast<const float4 *>(vrow + r * kD + 128 * jp + 4 * lane);
#pragma unroll
                        for (int eh = 0; eh < 2; ++eh) {
                            const float4 qa = wb[(4 * jp + 2 * eh) * 32];
                            const float4 qb = wb[(4 * jp + 2 * eh + 1) * 32];
#pragma unroll
                            for (int r = 0; r < NR; ++r) {
                                const float va = eh ? v4[r].z : v4[r].x;
                                const float vb = eh ? v4[r].w : v4[r].y;
                                const float da = ex2_approx(fminf(fmaf(a[r], gw[r][4 * jp + 2 * eh], qa.x), 60.0f)) + 1.0f;
                                const float db = ex2_approx(fminf(fmaf(a[r], gw[r][4 * jp + 2 * eh + 1], qb.x), 60.0f)) + 1.0f;
                                const float ri = rcp_approx(da * db);
                                accum5(acc[r], fmaf(-(va * oma[r]), ri * db, va), qa);
                                accum5(acc[r], fmaf(-(vb * oma[r]), ri * da, vb), qb);
                            }
                        }
                    }
                    {   // tail slot: dims 384 + lane, lanes 0..15 (v = gw = 0 elsewhere, address clamped)
                        const bool in = lane < 16;
                        const float4 q = wb[in ? 384 : 0];
#pragma unroll
                        for (int r = 0; r < NR; ++r) {
                            const float vv = in ? vrow[r * kD + 384 + lane] : 0.0f;
                            const float e = ex2_approx(fminf(fmaf(a[r], gw[r][12], q.x), 60.0f));
                            accum5(acc[r], fmaf(-(vv * oma[r]), rcp_approx(e + 1.0f), vv), q);
                        }
                    }
                    // split butterfly: 4x5 partial sums -> lane group (lane>>3) ends up owning row (lane>>3)
                    float k2[2][5];
                    const bool hi16 = (lane & 16) != 0, hi8 = (lane & 8) != 0;
#pragma unroll
                    for (int rr = 0; rr < 2; ++rr)
#pragma unroll
                        for (int q = 0; q < 5; ++q) {
                            const float send = hi16 ? acc[rr][q] : acc[rr + 2][q];
                            const float keep = hi16 ? acc[rr + 2][q] : acc[rr][q];
                            k2[rr][q] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
                        }
#pragma unroll
                    for (int q = 0; q < 5; ++q) {
                        const float send = hi8 ? k2[0][q] : k2[1][q];
                        const float keep = hi8 ? k2[1][q] : k2[0][q];
                        k1[q] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
                    }
#pragma unroll
                    for (int o = 4; o > 0; o >>= 1)
#pragma unroll
                        for (int q = 0; q < 5; ++q) k1[q] += __shfl_xor_sync(0xffffffffu, k1[q], o);
                };
                switch (nrows) {
                    case 4: rows(std::integral_constant<int, 4>{}); break;
                    case 3: rows(std::integral_constant<int, 3>{}); break;
                    case 2: rows(std::integral_constant<int, 2>{}); break;
                    case 1: rows(std::integral_constant<int, 1>{}); break;
                    default: break;
                }
                const int h = h0 + (lane >> 3);
                if ((lane & 7) == 0 && (lane >> 3) < nrows) {
                    const float *cs = S.cscal + c * 8;
                    const float mu = k1[0] * (1.0f / kD);
                    const float var = fmaxf(fmaf(-mu, mu, k1[1] * (1.0f / kD)), 0.0f);
                    const float rstd = rsqrtf(var + args.ln_eps);
                    S.lg_s[c * H + h] = fmaf(rstd, fmaf(-mu, cs[0], k1[2]), cs[3]);
                    S.y_s[c * H + h] = fmaf(rstd, fmaf(-mu, cs[1], k1[3]), cs[4]);
                    S.z_s[c * H + h] = fmaf(rstd, fmaf(-mu, cs[2], k1[4]), cs[5]);
                }
                if (has_next) {
#pragma unroll
                    for (int q = 0; q < 3; ++q) {
                        const int idx = tid + q * kThreads;
                        if (idx < kNW) {
                            const int which = idx / kD, d = idx - which * kD;
                            reinterpret_cast<float *>(S.wbuf + (buf ^ 1) * kD + wpos(d))[1 + which] = nvr[q] + nvt[q];
                        }
                    }
                }
                __syncthreads();
            }
        }

        // ---------------- phase 3: candidate-query pooling + lifetime-weighted dot ---------------
        for (int c = warp; c < cnt; c += kWarps) {
            const int P = S.cP[c];
            const int pz = P < H ? P : H;
            float m = -INFINITY;
            for (int hh = lane; hh < H; hh += 32) m = fmaxf(m, S.lg_s[c * H + hh]);
            m = warp_max(m);
            float l = 0.f, acc = 0.f, ms = 0.f;
            for (int hh = lane; hh < H; hh += 32) {
                const float e = __expf(S.lg_s[c * H + hh] - m);
                l += e;
                acc = fmaf(e, S.y_s[c * H + hh], acc);
                if (hh < pz) ms += S.z_s[c * H + hh];
            }
            l = warp_sum(l);
            acc = warp_sum(acc);
            ms = warp_sum(ms);
            float un = 0.f;
            if (P > H) {   // user-node rows take part in the GraphSAGE mean (userEncoders.py:121,153)
                int j = P - H - 1;
                j = j < C.user_nodes ? j : C.user_nodes - 1;
                const float *u = C.un_prefix + (size_t)j * kD;
                const float *hr = C.hist_rows + (size_t)S.cnews[c] * LIME_HIST_LD + LIME_HIST_VC;
                const float *tr = C.hist_tab + (size_t)S.ctab[c] * LIME_HTAB_LD;
                for (int d = lane; d < kD; d += 32) un = fmaf(hr[d] + tr[d], u[d], un);
                un = warp_sum(un);
            }
            if (lane == 0) {
                const float base = (ms + un) / (float)P + S.cscal[c * 8 + 6] + acc / l;
                args.scores[(long long)pair0 + c] = base * S.cw[c];
            }
            if constexpr (kExplain) {
                // contrib_h = w (alpha_h y_h + [h < min(P, H)] z_h / P), bias = w (un / P + b_l . c)
                const long long pair = (long long)pair0 + c;
                const float w = S.cw[c];
                if (lane == 0) {
                    ex.bias[pair] = w * (un / (float)P + S.cscal[c * 8 + 6]);
                    ex.weight[pair] = w;
                }
                for (int hh = lane; hh < H; hh += 32) {
                    const float al = __expf(S.lg_s[c * H + hh] - m) / l;
                    const float zp = hh < pz ? S.z_s[c * H + hh] / (float)P : 0.0f;
                    ex.alpha[pair * H + hh] = al;
                    ex.topic_attn[pair * H + hh] = S.a_s[c * H + hh];
                    ex.contrib[pair * H + hh] = w * fmaf(al, S.y_s[c * H + hh], zp);
                }
            }
        }
    }
}

}  // namespace lime

namespace lime {

int64_t score_exact_smem(int H, int TC) { return (int64_t)smem_carve(nullptr, nullptr, H, TC); }

template <bool kExplain>
static int launch_exact(const ScoreArgs &a, const ExplainOut &ex, int grid_limit, cudaStream_t st) {
    const int H = a.imp.max_history, TC = a.imp.tile_c;
    const size_t smem = smem_carve(nullptr, nullptr, H, TC);
    LIME_CHECK_ARG(smem <= 232448, "lime_score_impressions: (H=%d, tile_c=%d) needs %zu B of shared memory", H, TC, smem);
    LIME_CUDA(cudaMemsetAsync(a.work_counter, 0, sizeof(int32_t), st));
    int grid = num_sms();
    if (grid > grid_limit) grid = grid_limit;
    const int passes = (H + 31) / 32;
    if (passes <= 2) {
        LIME_CUDA(cudaFuncSetAttribute(score_kernel<2, kExplain>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        score_kernel<2, kExplain><<<grid, kThreads, smem, st>>>(a, ex);
    } else if (passes <= 4) {
        LIME_CUDA(cudaFuncSetAttribute(score_kernel<4, kExplain>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        score_kernel<4, kExplain><<<grid, kThreads, smem, st>>>(a, ex);
    } else {
        LIME_CUDA(cudaFuncSetAttribute(score_kernel<7, kExplain>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        score_kernel<7, kExplain><<<grid, kThreads, smem, st>>>(a, ex);
    }
    LIME_LAUNCH_CHECK("score_kernel");
    return 0;
}

// exact kernel over all units (unit_list == NULL) or over the device-side fallback list
int launch_score_exact(const ScoreArgs &a, int grid_limit, cudaStream_t st) {
    return launch_exact<false>(a, ExplainOut{}, grid_limit, st);
}

// process-wide scoring mode (lime_score_configure)
static int g_score_mode = 0;
static float g_score_tol = 1e-6f;

}  // namespace lime

using namespace lime;

extern "C" int64_t lime_score_smem_bytes(int32_t max_history, int32_t tile_c) {
    return (int64_t)smem_carve(nullptr, nullptr, max_history, tile_c);
}

extern "C" int64_t lime_score_scratch_ints(int32_t num_units) { return 4 + (int64_t)(num_units > 0 ? num_units : 0); }

extern "C" int32_t lime_score_tile_c(int32_t max_history) {
    if (max_history <= LIME_TC_MAX_HISTORY) return LIME_TC_TILE_C;
    for (int tc = 48; tc >= 8; tc -= 8)
        if (smem_carve(nullptr, nullptr, max_history, tc) <= 232448) return tc;
    return 0;
}

extern "C" int lime_score_configure(int32_t mode, float tolerance) {
    LIME_CHECK_ARG(mode >= 0 && mode <= 2, "lime_score_configure: mode %d not in {0,1,2}", mode);
    g_score_mode = mode;
    g_score_tol = tolerance;
    return 0;
}

extern "C" int lime_score_impressions(const LimeNewsCache *cache, const LimeImpressions *imp,
                                      int64_t pair_index_base, int32_t prefix_main,
                                      int64_t tail_start, int32_t prefix_tail, float *scores,
                                      int32_t *scratch, void *stream) {
    LIME_CHECK_ARG(cache && imp && scores && scratch, "lime_score_impressions: null argument");
    const int H = imp->max_history, TC = imp->tile_c;
    LIME_CHECK_ARG(H >= 1 && H <= 224, "lime_score_impressions: max_history %d not in [1,224]", H);
    LIME_CHECK_ARG(TC >= 1, "lime_score_impressions: tile_c %d < 1", TC);
    LIME_CHECK_ARG(cache->num_buckets >= 1 && cache->news_num >= 1, "lime_score_impressions: empty cache");
    // runtime batch larger than max_history + config.batch_size is an out-of-range gather in the
    // reference (userEncoders.py:94,153); reject it instead of reading past user_node_embedding
    LIME_CHECK_ARG(prefix_main >= 1 && prefix_main <= H + cache->user_nodes,
                   "lime_score_impressions: prefix_main %d not in [1, %d]", prefix_main, H + cache->user_nodes);
    LIME_CHECK_ARG(prefix_tail >= 1 && prefix_tail <= H + cache->user_nodes,
                   "lime_score_impressions: prefix_tail %d not in [1, %d]", prefix_tail, H + cache->user_nodes);
    if (imp->num_units <= 0) return 0;

    ScoreArgs a = {};
    a.cache = *cache;
    a.imp = *imp;
    a.pair_index_base = pair_index_base;
    a.tail_start = tail_start;
    a.prefix_main = prefix_main;
    a.prefix_tail = prefix_tail;
    a.bucket_scale = (float)((double)cache->num_buckets / 7.0);
    a.ln_eps = 1e-5f;
    a.scores = scores;
    a.work_counter = scratch;
    a.unit_list = nullptr;
    a.unit_list_count = nullptr;
    a.fallback_list = scratch + 4;
    a.fallback_count = scratch + 1;
    a.interp_tol = g_score_mode == 2 ? 0.0f : g_score_tol;
    cudaStream_t st = as_stream(stream);

    const bool tc_ok = g_score_mode != 1 && H <= LIME_TC_MAX_HISTORY && TC <= LIME_TC_TILE_C &&
                       cache->topic_table != nullptr && cache->num_topics >= 1 && cache->cand16 != nullptr &&
                       cache->ctab16 != nullptr && cache->news_meta != nullptr && cache->hist_vg != nullptr && cache->htab_vg != nullptr && cache->tc_tables_ok != 0 && cache->topic_logit_absmax <= 64.0f;
    if (!tc_ok) return launch_score_exact(a, imp->num_units, st);

    // fast path: interpolated gate + tcgen05 dots; units whose error bound exceeds the tolerance are
    // appended to a device-side list and re-scored by the exact kernel (usually an empty launch)
    int rc = launch_score_tc(a, st);
    if (rc != 0) return rc;
    a.work_counter = scratch + 2;
    a.unit_list = scratch + 4;
    a.unit_list_count = scratch + 1;
    return launch_score_exact(a, imp->num_units, st);
}

extern "C" int lime_explain_pairs(const LimeNewsCache *cache, const LimeImpressions *imp, int32_t prefix_main, float *scores,
                                  float *alpha, float *topic_attn, float *contrib, float *bias, float *weight, int32_t *scratch,
                                  void *stream) {
    LIME_CHECK_ARG(cache && imp && scores && alpha && topic_attn && contrib && bias && weight && scratch,
                   "lime_explain_pairs: null argument");
    const int H = imp->max_history, TC = imp->tile_c;
    LIME_CHECK_ARG(H >= 1 && H <= 224, "lime_explain_pairs: max_history %d not in [1,224]", H);
    LIME_CHECK_ARG(TC >= 1, "lime_explain_pairs: tile_c %d < 1", TC);
    LIME_CHECK_ARG(cache->num_buckets >= 1 && cache->news_num >= 1, "lime_explain_pairs: empty cache");
    LIME_CHECK_ARG(prefix_main >= 1 && prefix_main <= H + cache->user_nodes,
                   "lime_explain_pairs: prefix_main %d not in [1, %d]", prefix_main, H + cache->user_nodes);
    if (imp->num_units <= 0) return 0;

    ScoreArgs a = {};
    a.cache = *cache;
    a.imp = *imp;
    a.tail_start = 1LL << 62;
    a.prefix_main = prefix_main;
    a.prefix_tail = prefix_main;
    a.bucket_scale = (float)((double)cache->num_buckets / 7.0);
    a.ln_eps = 1e-5f;
    a.scores = scores;
    a.work_counter = scratch;
    const ExplainOut ex = {alpha, topic_attn, contrib, bias, weight};
    return launch_exact<true>(a, ex, imp->num_units, as_stream(stream));
}

// ---- histories longer than the tensor-core kernel's 56 slots (BASELINE.json configs[4]: history 100 / 200) ------------------
extern "C" int64_t lime_score_long_scratch_ints(int32_t chunked_units, int32_t orig_units) {
    return lime_score_scratch_ints(chunked_units) + 32 + (int64_t)(orig_units > 0 ? orig_units : 0);
}
extern "C" int64_t lime_score_long_work_floats(int64_t num_pairs, int32_t max_history, int32_t chunks) {
    if (num_pairs <= 0 || chunks <= 0) return 0;
    return (num_pairs * (int64_t)max_history + 3) / 4 * 4 + 4 * num_pairs * chunks + 2 * num_pairs;
}

namespace lime {
namespace {
__global__ void long_fallback_setup_kernel(const int *fallback_count, int orig_units, int *count_out, int *list_out) {
    const int n = *fallback_count > 0 ? orig_units : 0;       // any flagged chunk unit: the exact kernel re-scores the whole set
    if (blockIdx.x == 0 && threadIdx.x == 0) *count_out = n;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < orig_units; i += gridDim.x * blockDim.x) list_out[i] = i;
}
}  // namespace
}  // namespace lime

extern "C" int lime_score_impressions_long(const LimeNewsCache *cache, const LimeImpressions *imp, const LimeImpressions *chunked,
                                           int32_t chunks, int64_t num_pairs, int32_t num_impressions, int64_t pair_index_base, int32_t prefix_main,
                                           int64_t tail_start, int32_t prefix_tail, float *scores, int32_t *scratch, float *work,
                                           void *stream) {
    using namespace lime;
    LIME_CHECK_ARG(cache && imp && chunked && scores && scratch && work, "lime_score_impressions_long: null argument");
    const int H = imp->max_history, Hc = chunked->max_history;
    LIME_CHECK_ARG(chunks >= 2 && Hc >= 1 && Hc <= LIME_TC_MAX_HISTORY && Hc * chunks == H && H <= 224,
                   "lime_score_impressions_long: history %d is not %d chunks of %d <= %d slots", H, chunks, Hc, LIME_TC_MAX_HISTORY);
    LIME_CHECK_ARG(prefix_main >= 1 && prefix_main <= H + cache->user_nodes && prefix_tail >= 1 && prefix_tail <= H + cache->user_nodes,
                   "lime_score_impressions_long: prefix not in [1, %d]", H + cache->user_nodes);
    LIME_CHECK_ARG(cache->topic_table != nullptr && cache->num_topics >= 1 && cache->cand16 != nullptr && cache->ctab16 != nullptr &&
                       cache->news_meta != nullptr && cache->hist_vg != nullptr && cache->htab_vg != nullptr && cache->tc_tables_ok != 0 &&
                       cache->topic_logit_absmax <= 64.0f && g_score_mode != 1,
                   "lime_score_impressions_long: the cache does not carry the tensor-core operands (use lime_score_impressions)");
    LIME_CHECK_ARG(chunked->tile_c <= LIME_TC_TILE_C, "lime_score_impressions_long: chunked unit list built for tile %d", chunked->tile_c);
    if (imp->num_units <= 0 || num_pairs <= 0) return 0;
    cudaStream_t st = as_stream(stream);
    float *a_matrix = work;
    float4 *partial = reinterpret_cast<float4 *>(work + (num_pairs * (int64_t)H + 3) / 4 * 4);
    float2 *cbw = reinterpret_cast<float2 *>(reinterpret_cast<float *>(partial) + 4 * num_pairs * chunks);

    ScoreArgs o = {};                                   // the original set: attention pre-pass and the exact fallback
    o.cache = *cache;
    o.imp = *imp;
    o.pair_index_base = pair_index_base;
    o.tail_start = tail_start;
    o.prefix_main = prefix_main;
    o.prefix_tail = prefix_tail;
    o.bucket_scale = (float)((double)cache->num_buckets / 7.0);
    o.ln_eps = 1e-5f;
    o.scores = scores;
    if (int rc = launch_attention_long(o, a_matrix, chunks, Hc, num_pairs, st)) return rc;

    ScoreArgs a = o;                                    // the chunked set on the tensor-core kernel
    a.imp = *chunked;
    a.scores = nullptr;
    a.work_counter = scratch;
    a.fallback_list = scratch + 4;
    a.fallback_count = scratch + 1;
    a.interp_tol = g_score_mode == 2 ? 0.0f : g_score_tol;
    a.a_matrix = a_matrix;
    a.partial_out = partial;
    a.cbw_out = cbw;
    a.chunk_impressions = num_impressions;
    a.full_history = H;
    a.chunk_pairs = num_pairs;
    if (int rc = launch_score_tc(a, st)) return rc;
    if (int rc = launch_merge_long(o, partial, cbw, chunks, num_pairs, scores, st)) return rc;
    // a chunk unit the tensor-core kernel flagged (remainder bound, fp16 range, operand rows): the exact kernel re-scores the
    // whole original set (device-side decision, normally an empty launch)
    int32_t *tail = scratch + lime_score_scratch_ints(chunked->num_units);
    long_fallback_setup_kernel<<<64, 256, 0, st>>>(scratch + 1, imp->num_units, tail, tail + 32);
    LIME_LAUNCH_CHECK("long_fallback_setup_kernel");
    o.work_counter = scratch + 2;
    o.unit_list = tail + 32;
    o.unit_list_count = tail;
    o.fallback_list = nullptr;
    o.fallback_count = nullptr;
    return launch_score_exact(o, imp->num_units, st);
}
