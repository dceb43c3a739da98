// Training-mode forward and backward kernels of the CROWN user encoder + click score
// (userEncoders.py:101-175, layers.py:52-93, util.py:23-49) for the training layout: N = 1 + M candidates
// per sample share one history (model.py:171-181).  Unlike the eval path nothing is folded or cached: the
// weights change every step, so the dense layers are ordinary GEMMs (lime_linear / lime_gemm) and the
// kernels below are the non-GEMM pieces between them.  fp32, one CTA per sample unless noted.
#include "common.cuh"

namespace lime {

constexpr int kUD = LIME_D;             // 400
constexpr int kUHeads = LIME_CA_HEADS;  // 10
constexpr int kUHd = kUD / kUHeads;     // 40

// ---------------------------------------------------------------------------------------------
// Candidate-aware attention weights (layers.py:66-81):
//   S[hd][n][h] = Q_n[hd] . K_h[hd] / sqrt(D);  masked_fill(mask == 0, -1e9);  P = softmax_h(S)
//   P~ = dropout(P, p) (layers.py:36,74: nn.Dropout(0.2) on the attention weights; stateless mask of (seed, sample, index))
//   qw = softmax_n(||Q_n||_2);  agg[h] = sum_n qw_n sum_hd P~[hd][n][h];  a = softmax_h(agg)   (unmasked)
// Shared memory: Q [N][400], K [H][400], P [10*N][H], small vectors.
// ---------------------------------------------------------------------------------------------
struct CaSmem {
    float *Q, *K, *P, *qn, *qw, *agg, *a;
};
__device__ __forceinline__ CaSmem ca_carve(float *sm, int N, int H) {
    CaSmem s;
    s.Q = sm;
    s.K = s.Q + N * kUD;
    s.P = s.K + H * kUD;
    s.qn = s.P + kUHeads * N * H;
    s.qw = s.qn + N;
    s.agg = s.qw + N;
    s.a = s.agg + H;
    return s;
}
__host__ __device__ inline size_t ca_smem_floats(int N, int H) {
    return (size_t)N * kUD + (size_t)H * kUD + (size_t)kUHeads * N * H + 2 * N + 2 * H + 8;
}
// Dynamic shared memory both directions admit: the 227 KB opt-in less 1 KB for the backward's static dagg / dqw / red arrays.
// One limit for both, so that no (N, H) runs its forward and then fails in its backward.
constexpr size_t kCaSmemLimit = 232448 - 1024;

// forward pieces shared by the forward and backward kernels; on return P (before the dropout), qn, qw, agg, a are valid
__device__ void ca_forward(const CaSmem &s, const float *__restrict__ Qp, const float *__restrict__ Kp,
                           const uint8_t *__restrict__ mask, int N, int H, float scale, float p_drop, uint64_t seed,
                           uint64_t base_idx) {
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
    for (int i = tid; i < N * kUD; i += nt) s.Q[i] = Qp[i];
    for (int i = tid; i < H * kUD; i += nt) s.K[i] = Kp[i];
    __syncthreads();
    for (int idx = tid; idx < kUHeads * N * H; idx += nt) {
        const int h = idx % H, n = (idx / H) % N, hd = idx / (H * N);
        const float *q = s.Q + n * kUD + hd * kUHd, *k = s.K + h * kUD + hd * kUHd;
        float acc = 0.0f;
#pragma unroll 8
        for (int e = 0; e < kUHd; ++e) acc = fmaf(q[e], k[e], acc);
        s.P[idx] = mask[h] ? acc * scale : -1e9f;
    }
    for (int n = warp; n < N; n += nw) {
        float q2 = 0.0f;
        for (int e = lane; e < kUD; e += 32) q2 = fmaf(s.Q[n * kUD + e], s.Q[n * kUD + e], q2);
        q2 = warp_sum(q2);
        if (lane == 0) s.qn[n] = sqrtf(q2);
    }
    __syncthreads();
    for (int row = warp; row < kUHeads * N; row += nw) {           // softmax over h of every (head, candidate)
        float *p = s.P + row * H;
        float m = -INFINITY;
        for (int h = lane; h < H; h += 32) m = fmaxf(m, p[h]);
        m = warp_max(m);
        float l = 0.0f;
        for (int h = lane; h < H; h += 32) {
            const float e = expf(p[h] - m);
            p[h] = e;
            l += e;
        }
        l = 1.0f / warp_sum(l);
        for (int h = lane; h < H; h += 32) p[h] *= l;
    }
    if (warp == 0) {                                                // query weights: softmax over the candidates
        float m = -INFINITY;
        for (int n = lane; n < N; n += 32) m = fmaxf(m, s.qn[n]);
        m = warp_max(m);
        float l = 0.0f;
        for (int n = lane; n < N; n += 32) l += expf(s.qn[n] - m);
        l = warp_sum(l);
        for (int n = lane; n < N; n += 32) s.qw[n] = expf(s.qn[n] - m) / l;
    }
    __syncthreads();
    for (int h = tid; h < H; h += nt) {
        float acc = 0.0f;
        for (int n = 0; n < N; ++n) {
            float t = 0.0f;
            for (int hd = 0; hd < kUHeads; ++hd) {
                const int idx = (hd * N + n) * H + h;
                t += p_drop > 0.0f ? s.P[idx] * drop_scale(seed, base_idx + idx, p_drop) : s.P[idx];
            }
            acc = fmaf(s.qw[n], t, acc);
        }
        s.agg[h] = acc;
    }
    __syncthreads();
    if (warp == 0) {
        float m = -INFINITY;
        for (int h = lane; h < H; h += 32) m = fmaxf(m, s.agg[h]);
        m = warp_max(m);
        float l = 0.0f;
        for (int h = lane; h < H; h += 32) l += expf(s.agg[h] - m);
        l = warp_sum(l);
        for (int h = lane; h < H; h += 32) s.a[h] = expf(s.agg[h] - m) / l;
    }
    __syncthreads();
}

__global__ void __launch_bounds__(256)
ca_attn_fwd_kernel(const float *__restrict__ Qp, const float *__restrict__ Kp, const uint8_t *__restrict__ mask, int N, int H,
                   float scale, float p_drop, uint64_t seed, float *__restrict__ a_out) {
    extern __shared__ float sm[];
    const CaSmem s = ca_carve(sm, N, H);
    const int b = blockIdx.x;
    ca_forward(s, Qp + (size_t)b * N * kUD, Kp + (size_t)b * H * kUD, mask + (size_t)b * H, N, H, scale, p_drop, seed,
               (uint64_t)b * kUHeads * N * H);
    for (int h = threadIdx.x; h < H; h += blockDim.x) a_out[(size_t)b * H + h] = s.a[h];
}

__global__ void __launch_bounds__(256)
ca_attn_bwd_kernel(const float *__restrict__ Qp, const float *__restrict__ Kp, const uint8_t *__restrict__ mask, int N, int H,
                   float scale, float p_drop, uint64_t seed, const float *__restrict__ da, float *__restrict__ dQp,
                   float *__restrict__ dKp) {
    extern __shared__ float sm[];
    const CaSmem s = ca_carve(sm, N, H);
    __shared__ float dagg[64], dqw[64], red[2];
    const int b = blockIdx.x;
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
    const uint64_t base_idx = (uint64_t)b * kUHeads * N * H;
    ca_forward(s, Qp + (size_t)b * N * kUD, Kp + (size_t)b * H * kUD, mask + (size_t)b * H, N, H, scale, p_drop, seed, base_idx);
    const float *dab = da + (size_t)b * H;
    // a = softmax(agg):  dagg = a (da - sum a da)
    if (warp == 0) {
        float t = 0.0f;
        for (int h = lane; h < H; h += 32) t = fmaf(s.a[h], dab[h], t);
        t = warp_sum(t);
        for (int h = lane; h < H; h += 32) dagg[h] = s.a[h] * (dab[h] - t);
    }
    __syncthreads();
    // dqw_n = sum_h dagg_h sum_hd P[hd][n][h]
    for (int n = warp; n < N; n += nw) {
        float t = 0.0f;
        for (int h = lane; h < H; h += 32) {
            float ps = 0.0f;
            for (int hd = 0; hd < kUHeads; ++hd) {
                const int idx = (hd * N + n) * H + h;
                ps += p_drop > 0.0f ? s.P[idx] * drop_scale(seed, base_idx + idx, p_drop) : s.P[idx];
            }
            t = fmaf(dagg[h], ps, t);
        }
        t = warp_sum(t);
        if (lane == 0) dqw[n] = t;
    }
    __syncthreads();
    if (tid == 0) {
        float t = 0.0f;
        for (int n = 0; n < N; ++n) t = fmaf(s.qw[n], dqw[n], t);
        red[0] = t;
    }
    __syncthreads();
    // dS[hd][n][h] = P (dP - sum_h dP P) * scale with dP = dagg_h qw_n * dropout scale  (in place of P)
    for (int row = warp; row < kUHeads * N; row += nw) {
        const int n = row % N;
        float *p = s.P + row * H;
        float t = 0.0f;
        for (int h = lane; h < H; h += 32) {
            const float m = p_drop > 0.0f ? drop_scale(seed, base_idx + row * H + h, p_drop) : 1.0f;
            t = fmaf(dagg[h] * s.qw[n] * m, p[h], t);
        }
        t = warp_sum(t);
        // masked_fill: no gradient reaches the logits of masked history slots (they are the constant -1e9)
        for (int h = lane; h < H; h += 32) {
            const float m = p_drop > 0.0f ? drop_scale(seed, base_idx + row * H + h, p_drop) : 1.0f;
            p[h] = mask[(size_t)b * H + h] ? p[h] * (dagg[h] * s.qw[n] * m - t) * scale : 0.0f;
        }
    }
    __syncthreads();
    // dQ_n = sum_h dS K_h (per head) + dqn_n Q_n / ||Q_n||,  dqn = qw (dqw - sum qw dqw)
    for (int idx = tid; idx < N * kUD; idx += nt) {
        const int n = idx / kUD, e = idx - n * kUD, hd = e / kUHd;
        const float *ds = s.P + (hd * N + n) * H;
        float acc = 0.0f;
        for (int h = 0; h < H; ++h) acc = fmaf(ds[h], s.K[h * kUD + e], acc);
        const float dqn = s.qw[n] * (dqw[n] - red[0]);
        if (s.qn[n] > 0.0f) acc = fmaf(dqn / s.qn[n], s.Q[idx], acc);
        dQp[(size_t)b * N * kUD + idx] = acc;
    }
    for (int idx = tid; idx < H * kUD; idx += nt) {
        const int h = idx / kUD, e = idx - h * kUD, hd = e / kUHd;
        float acc = 0.0f;
        for (int n = 0; n < N; ++n) acc = fmaf(s.P[(hd * N + n) * H + h], s.Q[n * kUD + e], acc);
        dKp[(size_t)b * H * kUD + idx] = acc;
    }
}

// ---------------------------------------------------------------------------------------------
// wc = a * v (row scale, layers.py:84) and its backward
// ---------------------------------------------------------------------------------------------
__global__ void row_scale_fwd_kernel(const float *__restrict__ v, const float *__restrict__ a, int64_t rows, int d,
                                     float *__restrict__ out) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < rows * d) out[idx] = v[idx] * a[idx / d];
}
// one warp per row: dv = a dwc, da = sum_d dwc v
__global__ void __launch_bounds__(256)
row_scale_bwd_kernel(const float *__restrict__ v, const float *__restrict__ a, const float *__restrict__ dwc, int64_t rows, int d,
                     float *__restrict__ dv, float *__restrict__ da) {
    const int lane = threadIdx.x & 31;
    const int64_t r = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (r >= rows) return;
    const float ar = a[r];
    float t = 0.0f;
    for (int c = lane; c < d; c += 32) {
        const float g = dwc[r * d + c];
        dv[r * d + c] = ar * g;
        t = fmaf(g, v[r * d + c], t);
    }
    t = warp_sum(t);
    if (lane == 0) da[r] = t;
}

// ---------------------------------------------------------------------------------------------
// o = sigmoid(z) wc + (1 - sigmoid(z)) v   (layers.py:87-88) and its backward
// ---------------------------------------------------------------------------------------------
__global__ void gate_mix_fwd_kernel(const float *__restrict__ z, const float *__restrict__ wc, const float *__restrict__ v,
                                    int64_t total, float *__restrict__ o) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const float g = 1.0f / (1.0f + expf(-z[i]));
    o[i] = g * wc[i] + (1.0f - g) * v[i];
}
__global__ void gate_mix_bwd_kernel(const float *__restrict__ z, const float *__restrict__ wc, const float *__restrict__ v,
                                    const float *__restrict__ dout, int64_t total, float *__restrict__ dz,
                                    float *__restrict__ dwc, float *__restrict__ dv) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const float g = 1.0f / (1.0f + expf(-z[i]));
    const float go = dout[i];
    dz[i] = go * (wc[i] - v[i]) * g * (1.0f - g);
    dwc[i] = go * g;
    dv[i] = go * (1.0f - g);
}

// ---------------------------------------------------------------------------------------------
// GraphSAGE mean over node indices 0..P-1 of [x_b (H rows) ; user-node rows]  (userEncoders.py:91-98,121,153):
//   m[b] = (sum_{h < min(P,H)} x[b,h] + sum_{j < P-H} un[j]) / P
// ---------------------------------------------------------------------------------------------
__global__ void sage_mean_fwd_kernel(const float *__restrict__ x, const float *__restrict__ un, int B, int H, int P, int d,
                                     float *__restrict__ m) {
    const int b = blockIdx.x;
    const int pz = P < H ? P : H, pu = P > H ? P - H : 0;
    for (int c = threadIdx.x; c < d; c += blockDim.x) {
        float s = 0.0f;
        for (int h = 0; h < pz; ++h) s += x[((size_t)b * H + h) * d + c];
        for (int j = 0; j < pu; ++j) s += un[(size_t)j * d + c];
        m[(size_t)b * d + c] = s / (float)P;
    }
}
// dx[b,h] = dm[b] / P for h < min(P,H) else 0;  dun[j] = sum_b dm[b] / P for j < P - H else 0
__global__ void sage_mean_bwd_kernel(const float *__restrict__ dm, int B, int H, int P, int d, int un_rows,
                                     float *__restrict__ dx, float *__restrict__ dun) {
    const int pz = P < H ? P : H, pu = P > H ? P - H : 0;
    const float inv = 1.0f / (float)P;
    const int64_t total = (int64_t)B * H * d;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(idx % d);
        const int h = (int)((idx / d) % H);
        const int b = (int)(idx / ((int64_t)d * H));
        dx[idx] = h < pz ? dm[(size_t)b * d + c] * inv : 0.0f;
    }
    if (blockIdx.x == 0) {
        for (int idx = threadIdx.x; idx < un_rows * d; idx += blockDim.x) {
            const int j = idx / d, c = idx - j * d;
            float s = 0.0f;
            if (j < pu)
                for (int b = 0; b < B; ++b) s += dm[(size_t)b * d + c];
            dun[idx] = s * inv;
        }
    }
}

// g[b,h] = r[b,h] + l[b]  and  dl[b] = sum_h dg[b,h]
__global__ void add_row_bcast_kernel(const float *__restrict__ r, const float *__restrict__ l, int64_t rows, int H, int d,
                                     float *__restrict__ g) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows * d) return;
    const int64_t row = idx / d;
    g[idx] = r[idx] + l[(row / H) * d + (idx - row * d)];
}
__global__ void sum_over_h_kernel(const float *__restrict__ dg, int B, int H, int d, float *__restrict__ dl) {
    const int b = blockIdx.x;
    for (int c = threadIdx.x; c < d; c += blockDim.x) {
        float s = 0.0f;
        for (int h = 0; h < H; ++h) s += dg[((size_t)b * H + h) * d + c];
        dl[(size_t)b * d + c] = s;
    }
}

// ---------------------------------------------------------------------------------------------
// Candidate-query pooling (userEncoders.py:158-171): logits[n][h] = Kg[h] . q[n] / sqrt(A),
// alpha = softmax_h (unmasked), u[n] = sum_h alpha[n][h] g[h].  One CTA per sample, one warp per candidate.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
pool_fwd_kernel(const float *__restrict__ Kg, const float *__restrict__ q, const float *__restrict__ g, int N, int H, float scale,
                float *__restrict__ u, float *__restrict__ alpha_out) {
    extern __shared__ float sm[];      // alpha [N][H]
    const int b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const float *Kb = Kg + (size_t)b * H * kUD, *gb = g + (size_t)b * H * kUD;
    for (int n = warp; n < N; n += nw) {
        const float *qn = q + ((size_t)b * N + n) * kUD;
        float *al = sm + n * H;
        float m = -INFINITY;
        for (int h = 0; h < H; ++h) {
            float t = 0.0f;
            for (int e = lane; e < kUD; e += 32) t = fmaf(Kb[h * kUD + e], qn[e], t);
            t = warp_sum(t) * scale;
            if (lane == 0) al[h] = t;
            m = fmaxf(m, t);
        }
        __syncwarp();
        float l = 0.0f;
        for (int h = lane; h < H; h += 32) {
            const float e = expf(al[h] - m);
            al[h] = e;
            l += e;
        }
        l = 1.0f / warp_sum(l);
        __syncwarp();
        for (int h = lane; h < H; h += 32) {
            al[h] *= l;
            alpha_out[((size_t)b * N + n) * H + h] = al[h];
        }
        __syncwarp();
        for (int e = lane; e < kUD; e += 32) {
            float t = 0.0f;
            for (int h = 0; h < H; ++h) t = fmaf(al[h], gb[h * kUD + e], t);
            u[((size_t)b * N + n) * kUD + e] = t;
        }
    }
}
// du [B,N,400] -> dKg [B,H,400], dq [B,N,400], dg [B,H,400] (all overwritten)
__global__ void __launch_bounds__(256)
pool_bwd_kernel(const float *__restrict__ Kg, const float *__restrict__ q, const float *__restrict__ g,
                const float *__restrict__ alpha, const float *__restrict__ du, int N, int H, float scale,
                float *__restrict__ dKg, float *__restrict__ dq, float *__restrict__ dg) {
    extern __shared__ float sm[];      // dlogit [N][H]
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
    const float *Kb = Kg + (size_t)b * H * kUD, *gb = g + (size_t)b * H * kUD;
    for (int n = warp; n < N; n += nw) {
        const float *dun = du + ((size_t)b * N + n) * kUD;
        const float *al = alpha + ((size_t)b * N + n) * H;
        float *dl = sm + n * H;
        float dot = 0.0f;
        for (int h = 0; h < H; ++h) {
            float t = 0.0f;
            for (int e = lane; e < kUD; e += 32) t = fmaf(dun[e], gb[h * kUD + e], t);
            t = warp_sum(t);                              // d alpha[h]
            if (lane == 0) dl[h] = t;
            dot = fmaf(al[h], t, dot);
        }
        __syncwarp();
        for (int h = lane; h < H; h += 32) dl[h] = al[h] * (dl[h] - dot) * scale;
        __syncwarp();
        const float *qn = q + ((size_t)b * N + n) * kUD;
        for (int e = lane; e < kUD; e += 32) {
            float t = 0.0f;
            for (int h = 0; h < H; ++h) t = fmaf(dl[h], Kb[h * kUD + e], t);
            dq[((size_t)b * N + n) * kUD + e] = t;
        }
        (void)qn;
    }
    __syncthreads();
    for (int idx = tid; idx < H * kUD; idx += blockDim.x) {
        const int h = idx / kUD, e = idx - h * kUD;
        float tk = 0.0f, tg = 0.0f;
        for (int n = 0; n < N; ++n) {
            tk = fmaf(sm[n * H + h], q[((size_t)b * N + n) * kUD + e], tk);
            tg = fmaf(alpha[((size_t)b * N + n) * H + h], du[((size_t)b * N + n) * kUD + e], tg);
        }
        dKg[(size_t)b * H * kUD + idx] = tk;
        dg[(size_t)b * H * kUD + idx] = tg;
    }
}

// ---------------------------------------------------------------------------------------------
// click score with remaining-lifetime weighting (util.py:23-49): s = (u . c) w(r)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float lifetime_w(float r, float alpha, float beta, int use_w, int use_pen) {
    if (!use_w) return 1.0f;
    if (use_pen) {
        const float s = __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-__fmul_rn(alpha, r))));
        const float pos = (r >= 0.0f) ? 1.0f : 0.0f, neg = (r < 0.0f) ? 1.0f : 0.0f;
        return __fadd_rn(__fmul_rn(pos, s), __fmul_rn(__fmul_rn(neg, beta), s));
    }
    return __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-__fmul_rn(alpha, fabsf(r)))));
}
__global__ void __launch_bounds__(256)
score_fwd_kernel(const float *__restrict__ u, const float *__restrict__ c, const float *__restrict__ rem, int64_t rows,
                 float alpha, float beta, int use_w, int use_pen, float *__restrict__ s, float *__restrict__ w_out) {
    const int lane = threadIdx.x & 31;
    const int64_t r = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (r >= rows) return;
    float t = 0.0f;
    for (int e = lane; e < kUD; e += 32) t = fmaf(u[r * kUD + e], c[r * kUD + e], t);
    t = warp_sum(t);
    if (lane == 0) {
        const float w = lifetime_w(rem[r], alpha, beta, use_w, use_pen);
        w_out[r] = w;
        s[r] = t * w;
    }
}
__global__ void score_bwd_kernel(const float *__restrict__ u, const float *__restrict__ c, const float *__restrict__ w,
                                 const float *__restrict__ ds, int64_t rows, float *__restrict__ du, float *__restrict__ dc) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows * kUD) return;
    const int64_t r = idx / kUD;
    const float gsc = ds[r] * w[r];
    du[idx] = gsc * c[idx];
    dc[idx] = gsc * u[idx];
}

}  // namespace lime

using namespace lime;

static inline unsigned blocks_for(int64_t total, int per) { return (unsigned)((total + per - 1) / per); }

extern "C" int lime_ca_attention_fwd(const float *Qp, const float *Kp, const uint8_t *mask, int32_t B, int32_t N, int32_t H,
                                     float p_drop, uint64_t seed, float *a, void *stream) {
    LIME_CHECK_ARG(Qp && Kp && mask && a, "lime_ca_attention_fwd: null argument");
    LIME_CHECK_ARG(N >= 1 && N <= 64 && H >= 1 && H <= 64, "lime_ca_attention_fwd: N=%d, H=%d must be in [1,64]", N, H);
    if (B <= 0) return 0;
    const size_t smem = sizeof(float) * ca_smem_floats(N, H);
    LIME_CHECK_ARG(smem <= kCaSmemLimit, "lime_ca_attention_fwd: N=%d, H=%d needs %zu B of shared memory", N, H, smem);
    LIME_CUDA(cudaFuncSetAttribute(ca_attn_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ca_attn_fwd_kernel<<<B, 256, smem, as_stream(stream)>>>(Qp, Kp, mask, N, H, 1.0f / sqrtf((float)kUD), p_drop, seed, a);
    LIME_LAUNCH_CHECK("ca_attn_fwd_kernel");
    return 0;
}

extern "C" int lime_ca_attention_bwd(const float *Qp, const float *Kp, const uint8_t *mask, int32_t B, int32_t N, int32_t H,
                                     float p_drop, uint64_t seed, const float *da, float *dQp, float *dKp, void *stream) {
    LIME_CHECK_ARG(Qp && Kp && mask && da && dQp && dKp, "lime_ca_attention_bwd: null argument");
    LIME_CHECK_ARG(N >= 1 && N <= 64 && H >= 1 && H <= 64, "lime_ca_attention_bwd: N=%d, H=%d must be in [1,64]", N, H);
    if (B <= 0) return 0;
    const size_t smem = sizeof(float) * ca_smem_floats(N, H);
    LIME_CHECK_ARG(smem <= kCaSmemLimit, "lime_ca_attention_bwd: N=%d, H=%d needs %zu B of shared memory", N, H, smem);
    LIME_CUDA(cudaFuncSetAttribute(ca_attn_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ca_attn_bwd_kernel<<<B, 256, smem, as_stream(stream)>>>(Qp, Kp, mask, N, H, 1.0f / sqrtf((float)kUD), p_drop, seed, da, dQp, dKp);
    LIME_LAUNCH_CHECK("ca_attn_bwd_kernel");
    return 0;
}

extern "C" int lime_row_scale_fwd(const float *v, const float *a, int64_t rows, int d, float *out, void *stream) {
    LIME_CHECK_ARG(v && a && out, "lime_row_scale_fwd: null argument");
    if (rows <= 0) return 0;
    row_scale_fwd_kernel<<<blocks_for(rows * d, 256), 256, 0, as_stream(stream)>>>(v, a, rows, d, out);
    LIME_LAUNCH_CHECK("row_scale_fwd_kernel");
    return 0;
}
extern "C" int lime_row_scale_bwd(const float *v, const float *a, const float *dwc, int64_t rows, int d, float *dv, float *da,
                                  void *stream) {
    LIME_CHECK_ARG(v && a && dwc && dv && da, "lime_row_scale_bwd: null argument");
    if (rows <= 0) return 0;
    row_scale_bwd_kernel<<<blocks_for(rows, 8), 256, 0, as_stream(stream)>>>(v, a, dwc, rows, d, dv, da);
    LIME_LAUNCH_CHECK("row_scale_bwd_kernel");
    return 0;
}

extern "C" int lime_gate_mix_fwd(const float *z, const float *wc, const float *v, int64_t total, float *o, void *stream) {
    LIME_CHECK_ARG(z && wc && v && o, "lime_gate_mix_fwd: null argument");
    if (total <= 0) return 0;
    gate_mix_fwd_kernel<<<blocks_for(total, 256), 256, 0, as_stream(stream)>>>(z, wc, v, total, o);
    LIME_LAUNCH_CHECK("gate_mix_fwd_kernel");
    return 0;
}
extern "C" int lime_gate_mix_bwd(const float *z, const float *wc, const float *v, const float *dout, int64_t total, float *dz,
                                 float *dwc, float *dv, void *stream) {
    LIME_CHECK_ARG(z && wc && v && dout && dz && dwc && dv, "lime_gate_mix_bwd: null argument");
    if (total <= 0) return 0;
    gate_mix_bwd_kernel<<<blocks_for(total, 256), 256, 0, as_stream(stream)>>>(z, wc, v, dout, total, dz, dwc, dv);
    LIME_LAUNCH_CHECK("gate_mix_bwd_kernel");
    return 0;
}

extern "C" int lime_sage_mean_fwd(const float *x, const float *un, int32_t B, int32_t H, int32_t P, int32_t un_rows, float *m,
                                  void *stream) {
    LIME_CHECK_ARG(x && un && m, "lime_sage_mean_fwd: null argument");
    // a runtime batch larger than H + config.batch_size indexes past user_node_embedding in the reference
    LIME_CHECK_ARG(P >= 1 && P <= H + un_rows, "lime_sage_mean_fwd: prefix %d not in [1, %d]", P, H + un_rows);
    if (B <= 0) return 0;
    sage_mean_fwd_kernel<<<B, 128, 0, as_stream(stream)>>>(x, un, B, H, P, kUD, m);
    LIME_LAUNCH_CHECK("sage_mean_fwd_kernel");
    return 0;
}
extern "C" int lime_sage_mean_bwd(const float *dm, int32_t B, int32_t H, int32_t P, int32_t un_rows, float *dx, float *dun,
                                  void *stream) {
    LIME_CHECK_ARG(dm && dx && dun, "lime_sage_mean_bwd: null argument");
    LIME_CHECK_ARG(P >= 1 && P <= H + un_rows, "lime_sage_mean_bwd: prefix %d not in [1, %d]", P, H + un_rows);
    if (B <= 0) return 0;
    unsigned blocks = blocks_for((int64_t)B * H * kUD, 256);
    if (blocks > 4096) blocks = 4096;
    sage_mean_bwd_kernel<<<blocks, 256, 0, as_stream(stream)>>>(dm, B, H, P, kUD, un_rows, dx, dun);
    LIME_LAUNCH_CHECK("sage_mean_bwd_kernel");
    return 0;
}

extern "C" int lime_add_row_bcast(const float *r, const float *l, int64_t rows, int32_t H, int d, float *g, void *stream) {
    LIME_CHECK_ARG(r && l && g && H >= 1, "lime_add_row_bcast: bad argument");
    if (rows <= 0) return 0;
    add_row_bcast_kernel<<<blocks_for(rows * d, 256), 256, 0, as_stream(stream)>>>(r, l, rows, H, d, g);
    LIME_LAUNCH_CHECK("add_row_bcast_kernel");
    return 0;
}
extern "C" int lime_sum_over_h(const float *dg, int32_t B, int32_t H, int d, float *dl, void *stream) {
    LIME_CHECK_ARG(dg && dl, "lime_sum_over_h: null argument");
    if (B <= 0) return 0;
    sum_over_h_kernel<<<B, 128, 0, as_stream(stream)>>>(dg, B, H, d, dl);
    LIME_LAUNCH_CHECK("sum_over_h_kernel");
    return 0;
}

extern "C" int lime_pool_fwd(const float *Kg, const float *q, const float *g, int32_t B, int32_t N, int32_t H, float *u,
                             float *alpha, void *stream) {
    LIME_CHECK_ARG(Kg && q && g && u && alpha, "lime_pool_fwd: null argument");
    LIME_CHECK_ARG(N >= 1 && H >= 1 && (size_t)N * H * 4 <= 160000, "lime_pool_fwd: N=%d, H=%d too large", N, H);
    if (B <= 0) return 0;
    const size_t smem = sizeof(float) * (size_t)N * H;
    if (smem > 48000) LIME_CUDA(cudaFuncSetAttribute(pool_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    pool_fwd_kernel<<<B, 256, smem, as_stream(stream)>>>(Kg, q, g, N, H, 1.0f / sqrtf((float)kUD), u, alpha);
    LIME_LAUNCH_CHECK("pool_fwd_kernel");
    return 0;
}
extern "C" int lime_pool_bwd(const float *Kg, const float *q, const float *g, const float *alpha, const float *du, int32_t B,
                             int32_t N, int32_t H, float *dKg, float *dq, float *dg, void *stream) {
    LIME_CHECK_ARG(Kg && q && g && alpha && du && dKg && dq && dg, "lime_pool_bwd: null argument");
    LIME_CHECK_ARG(N >= 1 && H >= 1 && (size_t)N * H * 4 <= 160000, "lime_pool_bwd: N=%d, H=%d too large", N, H);
    if (B <= 0) return 0;
    const size_t smem = sizeof(float) * (size_t)N * H;
    if (smem > 48000) LIME_CUDA(cudaFuncSetAttribute(pool_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    pool_bwd_kernel<<<B, 256, smem, as_stream(stream)>>>(Kg, q, g, alpha, du, N, H, 1.0f / sqrtf((float)kUD), dKg, dq, dg);
    LIME_LAUNCH_CHECK("pool_bwd_kernel");
    return 0;
}

extern "C" int lime_click_score_fwd(const float *u, const float *c, const float *remaining, int64_t rows, float alpha,
                                    float beta, int32_t use_weighting, int32_t use_expired_penalty, float *scores, float *w,
                                    void *stream) {
    LIME_CHECK_ARG(u && c && remaining && scores && w, "lime_click_score_fwd: null argument");
    if (rows <= 0) return 0;
    score_fwd_kernel<<<blocks_for(rows, 8), 256, 0, as_stream(stream)>>>(u, c, remaining, rows, alpha, beta, use_weighting,
                                                                         use_expired_penalty, scores, w);
    LIME_LAUNCH_CHECK("score_fwd_kernel");
    return 0;
}
extern "C" int lime_click_score_bwd(const float *u, const float *c, const float *w, const float *dscores, int64_t rows,
                                    float *du, float *dc, void *stream) {
    LIME_CHECK_ARG(u && c && w && dscores && du && dc, "lime_click_score_bwd: null argument");
    if (rows <= 0) return 0;
    score_bwd_kernel<<<blocks_for(rows * kUD, 256), 256, 0, as_stream(stream)>>>(u, c, w, dscores, rows, du, dc);
    LIME_LAUNCH_CHECK("score_bwd_kernel");
    return 0;
}
