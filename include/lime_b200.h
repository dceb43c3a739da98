/*
 * lime_b200.h — C ABI of liblime_b200.so: the B200 (sm_100a) implementation of LIME's scoring hot
 * path (reference: seongeunryu/lime-cikm25).
 *
 * The reference is pure Python/PyTorch: its "FFI" for this path is the set of nn.Module forward
 * calls on the path.  Each entry point below names the reference interface it replaces
 * (file:line in the reference tree).  INTEGRATION.md shows the ctypes stub a maintainer would add
 * to the reference's newsEncoders.py / userEncoders.py / util.py to bind them.
 *
 * Conventions
 *   - Every pointer is a DEVICE pointer unless its name starts with h_.  The caller owns all
 *     memory (in this repo: torch tensors); the library never allocates or frees device memory.
 *   - `stream` is a cudaStream_t passed as void*.  Calls enqueue work on it and return without
 *     synchronising.
 *   - Return value: 0 on success, non-zero on error; lime_last_error() describes the last error
 *     raised on the calling thread.  There is no CPU fallback: without a CUDA device every compute
 *     entry point fails.
 *   - fp32 everywhere (the reference never enables TF32/autocast, config.py:218-219); ids int32 as
 *     the reference's corpus arrays (corpus.py:361-368); masks one byte per element (torch.bool).
 *   - Matrices are row-major with an explicit leading dimension (elements, not bytes).
 */
#ifndef LIME_B200_H_
#define LIME_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LIME_B200_ABI_VERSION 8

/* Compile-time model geometry of the LIME-CROWN-CROWN configuration (config.py:54-91 defaults). */
#define LIME_D        400   /* lime_output_dim == news_embedding_dim == attention_dim          */
#define LIME_TOPIC    50    /* category_embedding_dim (topic representation width)             */
#define LIME_TOPIC_LD 52    /* topic width padded to a multiple of 4 floats                    */
#define LIME_CA_HEADS 10    /* CandidateAware_ClickedNewsAttention.num_heads, layers.py:22     */

/* Row layout of the per-news vector cache (floats).  See DESIGN.md "HBM layout".               */
#define LIME_HIST_LD   852  /* [ vc 0..399 | gw 400..799 | topic 800..851 ]                    */
#define LIME_HIST_VC   0
#define LIME_HIST_GW   400
#define LIME_HIST_T    800
#define LIME_HIST_GW_ABSMAX 851 /* max_d |gw[d]| of the row (bounds the gate interpolation error)     */
#define LIME_HIST_TOPIC_ID 850 /* int32 bit pattern: compact id of the news' (category, subCategory) pair */
#define LIME_CAND_LD   1720 /* [ w1 | w2 | w3 | scal(8) | tq 50x10 | qb 10 | pad 2 ]           */
#define LIME_CAND_W    0
#define LIME_CAND_SCAL 1200
#define LIME_CAND_TQ   1208
#define LIME_CAND_QB   1708
#define LIME_CAND_TOPIC_ID 1718 /* int32 bit pattern, same id as LIME_HIST_TOPIC_ID                 */
#define LIME_CAND_NFOLD 1207 /* columns produced by the folded GEMM: w1,w2,w3 + 7 scalars       */
#define LIME_CAND_ABSMAX 1207 /* max |w1 w2 w3| of the row, written by lime_split_f16_pairs (fp16 operand range check) */
#define LIME_META_LD 8      /* news_meta row: topic id | gw absmax | w absmax | B1 | B2 | B3 | cb | pad */
#define LIME_CAND16_SCALE 1024.0f /* cand16 / ctab16 hold scale * w (keeps the lo halves out of the fp16 subnormals) */
#define LIME_CAND16_LD 2400 /* fp16 elements per row of cand16 / ctab16: [hi | lo][k = w1 w2 w3][400] -- an operand-row triple is 3 consecutive 800-byte rows */
#define LIME_HTAB_LD   800  /* per (freshness bucket, lifetime bucket): [ T | gwT ]            */
#define LIME_CTAB_LD   1208 /* per bucket pair: [ w1T | w2T | w3T | scalT(8) ]                 */
/* Tensor-core scoring path (score_tc.cu): history rows per impression, candidates per work unit. */
#define LIME_TC_MAX_HISTORY 56
#define LIME_TC_TILE_C      39  /* candidates of a unit + its distinct (freshness, lifetime) bucket pairs <= 40 operand-row
                                   triples: the host sizes the units accordingly (engine.build_units), a unit that still does
                                   not fit is re-scored by the exact kernel */
#define LIME_TOPIC_TAB_LD   12  /* 10 head logits of a (candidate topic, history topic) pair, padded */
#define LIME_TC_MAX_TOPICS  1024

int         lime_abi_version(void);
const char *lime_last_error(void);
/* Number of CUDA devices visible; <= 0 means the product path cannot run. */
int         lime_device_count(void);
/* Kernels launched by this library (any thread of the process) since the last reset (bench.py's
 * gpu_launches).  */
int64_t     lime_launch_count(void);
void        lime_launch_count_reset(void);

/* ---- FreshnessEncoder.bucketize, newsEncoders.py:53-58 (bit-exact) --------------------------- */
int lime_bucketize(const float *seconds, int64_t n, int num_buckets, int32_t *buckets, void *stream);

/* ---- dense building blocks (torch.nn.Linear / F.linear on the path) --------------------------
 * C[m, n] = act( A[m, :k] . W[n, :k]^T + bias[n] ) + residual[m, n]
 * act: 0 none, 1 relu, 2 tanh.  bias / residual may be NULL.  k, lda, ldw must be multiples of 4
 * and A, W 16-byte aligned (pad with zeros).                                                     */
int lime_linear(const float *A, int64_t lda, const float *W, int64_t ldw, const float *bias,
                const float *residual, int64_t ldr, float *C, int64_t ldc,
                int64_t m, int n, int k, int act, void *stream);
/* Same contract, operands rounded to bf16 and multiplied on the tcgen05 tensor cores with fp32
 * accumulation in TMEM ("bf16 mode" of the north star; metrics-level parity).                    */
int lime_linear_bf16(const float *A, int64_t lda, const float *W, int64_t ldw, const float *bias,
                     const float *residual, int64_t ldr, float *C, int64_t ldc,
                     int64_t m, int n, int k, int act, void *stream);
/* The dense layer of "bf16 mode" on bf16 ACTIVATIONS (Stage A cache build): A [m, lda] and W [n, ldw] are bf16 with the
 * contraction length k padded to a multiple of 64 (<= 512) by zero columns, bias / residual fp32, C bf16 (c_is_bf16 != 0;
 * columns n..ldc-1 are written as zeros so that C can be the next layer's A) or fp32.  TMA-fed, W slice resident in shared
 * memory, two TMEM accumulators (csrc/gemm_tma.cu).  Replaces the same reference lines as lime_linear.                   */
int lime_linear_bf16_tma(const void *A, int64_t lda, const void *W, int64_t ldw, const float *bias, const float *residual,
                         int64_t ldr, void *C, int64_t ldc, int32_t c_is_bf16, int64_t m, int32_t n, int32_t k, int32_t act,
                         float alpha, int32_t ab_is_fp16, void *stream);
/* alpha scales the accumulator before bias / residual (C = act(alpha A . W^T + bias) + residual); ab_is_fp16 != 0: A and W are
 * fp16 instead of bf16 (the hi / lo pairs of the fp32x3 mode, pre-scaled by powers of two: alpha undoes the scaling). */
/* act | LIME_ACT_RES_FIRST: the residual joins the sum BEFORE the activation, C = act(A . W^T + bias + residual): the
 * accumulating passes of the three-pass bf16x3 layer (residual = C, in place). */
#define LIME_ACT_RES_FIRST 16
/* The fp32x3 dense layer in ONE launch (fp32x3 encoder mode of newsEncoders.py:244-247's GEMMs): A = Ahi + Alo and W = Whi + Wlo
 * are 16-bit pairs from lime_split_bf16_pairs (same lda / ldw for both images, k padded to a multiple of 64, both W images
 * resident: 2 k bn 2 B <= 160 KB), C = act(alpha (Alo Whi^T + Ahi Wlo^T + Ahi Whi^T) + bias) + residual in fp32; the three
 * products accumulate in one TMEM tile, small ones first (the tensor core truncates addends at the accumulator's exponent),
 * so C is written once (the three-pass form re-reads and re-writes it twice). */
int lime_linear_x3_tma(const void *Ahi, const void *Alo, int64_t lda, const void *Whi, const void *Wlo, int64_t ldw,
                       const float *bias, const float *residual, int64_t ldr, float *C, int64_t ldc, int64_t m, int32_t n,
                       int32_t k, int32_t act, float alpha, int32_t ab_is_fp16, void *stream);
/* The same layer with the result leaving as the NEXT fp32x3 layer's operand pair: out_scale * act(alpha (...) + bias) = hi + lo
 * (fp16, each [m, ld16], ld16 a multiple of 8, columns n..ld16-1 zero) -- the FFN hidden layer of newsEncoders.py:244-247 never
 * exists as an fp32 matrix and no lime_split_bf16_pairs pass re-reads it.  No residual. */
int lime_linear_x3_pairs_tma(const void *Ahi, const void *Alo, int64_t lda, const void *Whi, const void *Wlo, int64_t ldw,
                             const float *bias, void *Chi, void *Clo, int64_t ld16, float out_scale, int64_t m, int32_t n,
                             int32_t k, int32_t act, float alpha, int32_t ab_is_fp16, void *stream);
/* fp32 rows -> 16-bit pair hi = r16(scale x), lo = r16(scale x - hi), each [rows, ld16] with columns d..ld16-1 zero; fp16 pairs
 * (as_fp16 != 0: scale x = hi + lo to 2^-22, scale a power of two that keeps hi below 65504) or bf16 pairs (2^-17).
 * With the same split of W, x . W^T ~ xh . Wh^T + xl . Wh^T + xh . Wl^T reproduces the fp32 product on the tensor cores
 * (three lime_linear_bf16_tma passes accumulating in place): the "fp32x3" encoder mode.  lo may be NULL: only the rounded image
 * hi is written (the operand cast of the bf16 training GEMMs). */
int lime_split_bf16_pairs(const float *x, int64_t ldx, int64_t rows, int32_t d, void *hi, void *lo, int32_t ld16, float scale,
                          int32_t as_fp16, void *stream);
/* bf16 image of x (as lime_split_bf16_pairs with lo = NULL, scale 1) AND colsum[c] += sum_r x[r, c] in the same pass: the operand
 * cast of dZ and the bias gradient of an nn.Linear backward in bf16 training mode.  d, ldx multiples of 4, ld16 a multiple of 8
 * (<= 1024), x and colsum 16-byte aligned; colsum [d] is accumulated (zero it first). */
int lime_cast_bf16_colsum(const float *x, int64_t ldx, int64_t rows, int32_t d, void *out16, int32_t ld16, float *colsum,
                          void *stream);
/* Small general GEMM with arbitrary strides (weight folding, done once per checkpoint):
 * C[i*ldc + j] = alpha * sum_k A[i*sam + k*sak] * B[k*sbk + j*sbn]                                */
int lime_gemm_strided(const float *A, int64_t sam, int64_t sak, const float *B, int64_t sbk,
                      int64_t sbn, float *C, int64_t ldc, int m, int n, int k, float alpha,
                      void *stream);

/* ---- newsEncoders.CROWN.forward pieces, newsEncoders.py:302-373 ------------------------------ */
/* word_embedding(ids) + PositionalEncoding (:311-315, :806-828): out[r, :] = E[ids[r], :] + pe[r % T, :] */
int lime_embed_pe(const float *E, int64_t vocab, const int32_t *ids, int64_t rows, int T, int d,
                  const float *pe, float *out, void *stream);
/* lime_embed_pe with a second, bf16 image of every row: out16 [rows, ld16] (columns d..ld16-1 zero), the A operand of
 * lime_linear_bf16_tma; out stays the fp32 residual stream. */
int lime_embed_pe_bf16(const float *E, int64_t vocab, const int32_t *ids, int64_t rows, int T, int d, const float *pe,
                       float *out, void *out16, int32_t ld16, void *stream);
/* nn.MultiheadAttention core of the TransformerEncoderLayer (:244-247), no mask:
 * qkv [n_news*T, 3*d] (q | k | v) -> ctx [n_news*T, d], softmax(q k^T / sqrt(d/nhead)) v per head.
 * Supported: T in {32, 128}, d/nhead <= 32.                                                      */
int lime_mha(const float *qkv, float *ctx, int64_t n_news, int T, int d, int nhead, float p_drop, uint64_t seed,
             int64_t news0, void *stream);
/* the same on bf16 activations and the tensor cores (eval only): qkv [n_news*T, ldq] bf16 in the HEAD-PADDED layout
 * q | k | v, each nhead slices of 32 columns (d/nhead real ones, the rest exact zeros: permute and zero-pad the rows of
 * in_proj_weight / in_proj_bias) -> ctx [n_news*T, ldo] bf16 in the plain layout, columns d..ldo-1 zero */
int lime_mha_bf16(const void *qkv, int64_t ldq, void *ctx, int64_t ldo, int64_t n_news, int T, int d, int nhead, void *stream);
/* p_drop / seed: dropout on the attention weights (training; 0 in eval), stateless mask of (seed, news0 + news, head, i, j)
 * -- news0 is the global index of the call's first news, so a chunked call sees the mask of the whole batch */
/* nn.LayerNorm over the last dim (eps as given). */
int lime_layernorm(const float *x, int64_t ldx, const float *gamma, const float *beta, float *y,
                   int64_t ldy, int64_t rows, int d, float eps, void *stream);
/* lime_layernorm with a second, bf16 image of every row: y16 [rows, ld16] (columns d..ld16-1 zero) */
int lime_layernorm_bf16(const float *x, int64_t ldx, const float *gamma, const float *beta, float *y, int64_t ldy,
                        void *y16, int32_t ld16, int64_t rows, int d, float eps, void *stream);
/* fp32x3-mode twins of lime_embed_pe_bf16 / lime_layernorm_bf16: beside the fp32 row, the fp16 operand PAIR scale * x = hi + lo
 * (each [rows, ld16], columns d..ld16-1 zero) of the next lime_linear_x3_tma -- the producer writes it, no lime_split_bf16_pairs
 * pass re-reads the row. */
int lime_embed_pe_pairs(const float *E, int64_t vocab, const int32_t *ids, int64_t rows, int T, int d, const float *pe,
                        float *out, void *hi16, void *lo16, int32_t ld16, float scale, void *stream);
int lime_layernorm_pairs(const float *x, int64_t ldx, const float *gamma, const float *beta, float *y, int64_t ldy,
                         void *hi16, void *lo16, int32_t ld16, float scale, int64_t rows, int d, float eps, void *stream);
/* LayerNorm of every token followed by the unmasked mean over the T tokens of a news (:317,:321):
 * x [n_news*T, d] -> out[n, :d] (row stride ldo). */
int lime_layernorm_meanpool(const float *x, const float *gamma, const float *beta, float *out,
                            int64_t ldo, int64_t n_news, int T, int d, float eps, void *stream);
/* category_affine(category_embedding(c) || subCategory_embedding(s)) (:340-342 and
 * userEncoders.py:103-105,115-117): out[n, :50] (row stride ldo; columns 50..width-1 zeroed). */
int lime_topic_rep(const float *cat_emb, const float *sub_emb, const float *W, const float *b,
                   const int32_t *cat, const int32_t *sub, int64_t n, float *out, int64_t ldo,
                   int width, void *stream);
/* layers.Attention over the k intents (layers.py:285-300): pre = affine1(e) (before tanh),
 * e [n, k, D] -> out [n, D] (row stride ldo) = sum_k softmax_k(w2 . tanh(pre_k)) e_k.             */
int lime_intent_pool(const float *pre, const float *e, const float *w2, float *out, int64_t ldo,
                     int64_t n, int k, int D, void *stream);
/* similarity_compute + concat + feature_fusion (:297-300,:367-371):
 * content[n] = [ title | (cos(title, body)+1)/2 * body | cat_emb[c] | sub_emb[s] ]  (row stride ldo) */
int lime_content_fuse(const float *title, const float *body, const float *cat_emb,
                      const float *sub_emb, const int32_t *cat, const int32_t *sub, int64_t n, int D,
                      int cat_dim, int sub_dim, float *content, int64_t ldo, void *stream);
/* FreshnessEncoder embedding concat for every (freshness bucket, lifetime bucket) pair (:78-81):
 * out[bf*nb + bl] = [ Ef[bf] | El[bl] ]                                                           */
int lime_bucket_pairs(const float *Ef, const float *El, int num_buckets, int dim, float *out,
                      void *stream);

/* small helpers used while folding weights */
/* out[i * ldo] = max_j |M[i * ld + j]|,  j < cols */
int lime_row_absmax(const float *M, int64_t ld, int64_t rows, int cols, float *out, int64_t ldo, void *stream);
int lime_scale_rows(float *M, int64_t ld, const float *row_scale, float alpha, int rows, int cols,
                    void *stream);                         /* M[i,:] *= alpha * row_scale[i] (NULL -> 1) */
int lime_prefix_rows(float *M, int64_t ld, int rows, int cols, void *stream); /* inclusive prefix sum over rows */

/* ---- userEncoders.CROWN.forward + RemainingLifetimeWeighting (eval, one candidate per sample) --
 * Replaces, for a whole impression set at once, what compute_scores (util.py:88-112) obtains by
 * calling Model.forward (model.py:151-187) on batches of (user, candidate) pairs:
 *   CandidateAware_ClickedNewsAttention (layers.py:52-93) -> GraphSAGE mean aggregation
 *   (userEncoders.py:121,151-157) -> candidate-query pooling (:158-171) -> lifetime-weighted dot
 *   (util.py:23-49), on cached news vectors (the reference re-encodes 50 history news per pair).
 * The reference's result depends on the runtime mini-batch size through GraphSAGE
 * (SURVEY.md §8a row 10): a pair with global index g uses prefix length
 *   P = (g >= tail_start) ? prefix_tail : prefix_main,    g = pair_index_base + local pair index.
 */
typedef struct {
    /* per-news cache built by the Python host from the entry points above */
    const float *hist_rows;     /* [news_num, LIME_HIST_LD]                                      */
    const float *cand_rows;     /* [news_num, LIME_CAND_LD]                                      */
    const float *hist_tab;      /* [tab_replicas, nb*nb, LIME_HTAB_LD]: identical copies; the tensor-core kernel reads copy
                                   blockIdx % tab_replicas (every CTA gathers the same few hot rows at every stage: one copy
                                   serialises them in a handful of L2 slices), the exact kernel copy 0             */
    const float *cand_tab;      /* [nb*nb, LIME_CTAB_LD]                                         */
    const float *gate_bias;     /* [LIME_D]  -log2(e) * gate_proj.bias                           */
    const float *un_prefix;     /* [config.batch_size, LIME_D] prefix sums of lin_l(user_node_embedding) */
    const float *topic_table;   /* [num_topics, num_topics, LIME_TOPIC_TAB_LD] from lime_topic_pair_table,
                                   or NULL (then only the exact kernel can run)                      */
    const void  *cand16;        /* [news_num + tab_replicas*nb*nb, LIME_CAND16_LD] fp16: w1 w2 w3 of cand_rows as hi/lo pairs
                                   (lime_split_f16_pairs), FOLLOWED by tab_replicas copies of the nb*nb rows of ctab16 (one
                                   operand array for candidate and bucket-pair rows), or NULL (exact kernel only)      */
    const void  *ctab16;        /* [nb*nb, LIME_CAND16_LD] fp16: the same for cand_tab (source of the tail of cand16) */
    const float *news_meta;     /* [news_num, LIME_META_LD]: the scalars phase 0 of the tensor-core kernel needs, packed
                                   into one 32-byte sector per news (2 MB for 65k news: L2 resident) -- topic id (int32
                                   bits), gw absmax, w absmax, B1, B2, B3, cb, 0; or NULL (exact kernel only)   */
    const float *hist_vg;       /* [news_num, 2*LIME_D]: vc and gw of hist_rows interleaved in groups of 4 dims
                                   (v0..3 g0..3 v4..7 g4..7 ...), 32-byte aligned rows: one 256-bit load fetches both
                                   operands of 4 dims (tensor-core kernel only; NULL: exact kernel only)                */
    const float *htab_vg;       /* [tab_replicas, nb*nb, 2*LIME_D]: hist_tab in the same interleaved layout             */
    int32_t news_num;
    int32_t num_buckets;
    int32_t user_nodes;         /* config.batch_size (rows of user_node_embedding)               */
    int32_t num_topics;         /* distinct (category, subCategory) pairs registered in the cache */
    float   tab_gw_absmax;      /* max |gw| over hist_tab (same purpose as LIME_HIST_GW_ABSMAX)   */
    float   sigmoid_alpha;      /* config.sigmoid_scaling_alpha                                  */
    float   penalty_beta;       /* config.penalty_scaling_beta                                   */
    int32_t use_lifetime_weighting; /* config.use_remaining_lifetime_weighting                   */
    int32_t use_expired_penalty;    /* config.use_expired_penalty                                */
    float   topic_logit_absmax; /* max |log2(entry)| of topic_table (entries are exponentials of the head logits): the tensor-core
                                   path runs its softmax without a max pass and requires this <= 64   */
    int32_t tc_tables_ok;       /* nonzero: ctab16 holds no value beyond the fp16 operand range      */
    int32_t tab_replicas;       /* copies of the bucket-pair tables in hist_tab and in the tail of cand16 (>= 1) */
} LimeNewsCache;

typedef struct {
    /* impression-major inputs (dataset.py:192-227 layout, candidates flattened) */
    const int32_t *hist_news;   /* [I, H] row index into the cache, padding = 0                  */
    const uint8_t *hist_mask;   /* [I, H]                                                        */
    const float   *hist_fresh;  /* [I, H] seconds                                                */
    const float   *hist_life;   /* [I, H] seconds                                                */
    const int32_t *cand_news;   /* [P]                                                           */
    const float   *cand_fresh;  /* [P]                                                           */
    const float   *cand_life;   /* [P]                                                           */
    const float   *cand_remaining; /* [P] remaining lifetime handed to RemainingLifetimeWeighting, or
                                      NULL: cand_life - cand_fresh (lifetime_type='user_topic',
                                      util.py:103-104)                                             */
    /* work units: consecutive candidates of one impression, at most tile_c each */
    const int32_t *unit_imp;    /* [U] impression of the unit                                    */
    const int32_t *unit_pair0;  /* [U] first (local) pair index                                  */
    const int32_t *unit_count;  /* [U] number of candidates, 1..tile_c                           */
    int32_t num_units;
    int32_t max_history;        /* H                                                             */
    int32_t tile_c;             /* capacity the unit list was built for                          */
} LimeImpressions;

/* scratch: caller-owned int32 device buffer of lime_score_scratch_ints(num_units) elements
 * (work counters + the list of units the fast path hands to the exact kernel); contents are
 * overwritten by every call.
 *
 * Two kernels implement the same arithmetic:
 *   - exact   (score.cu): every (candidate, history row) gate evaluated element by element; any H <= 224.
 *   - tensor  (score_tc.cu, H <= LIME_TC_MAX_HISTORY): history slots with the same (news, bucket pair, mask) are
 *     deduplicated; per unique row the gated vector and its derivative in the attention weight a are evaluated
 *     once, at the centre of a's range over the unit's candidates (economised second-order expansion), the 3 dots
 *     with every candidate are tcgen05 MMAs on fp16 hi/lo pairs (candidate side pre-split in cand16 / ctab16,
 *     the unit's distinct bucket-pair rows as extra operand rows, fp32 accumulation in TMEM), and each pair
 *     evaluates the expansion at its own a.  A unit whose a-spread makes the remainder bound exceed the
 *     tolerance, that holds an operand beyond the fp16 range, or has more distinct bucket pairs than spare
 *     operand rows, is re-scored by the exact kernel in the same call.
 * lime_score_configure(mode, tolerance): mode 0 = tensor path with exact fallback (default,
 * tolerance 1e-6 on the gate), 1 = exact only, 2 = tensor path with every unit forced through the
 * fallback (tests).  Process-wide. */
/* sizeof() of the two argument structs as this library was compiled (binding self-check). */
int64_t lime_sizeof_news_cache(void);
int64_t lime_sizeof_impressions(void);

/* Histories longer than LIME_TC_MAX_HISTORY slots on the tensor-core kernel (BASELINE.json configs[4]: history 100 / 200).
 * `imp` is the original set (H = imp->max_history <= 224, its unit list serves the exact-kernel fallback); `chunked` holds the
 * same impressions cut into `chunks` pieces of Hc = H / chunks <= LIME_TC_MAX_HISTORY slots: pseudo-impression k * num_impressions
 * + i = slots [k Hc, (k + 1) Hc) of impression i, candidate arrays replicated chunk-major (pair k * num_pairs + p), unit list
 * planned for the tensor-core kernel.  A pre-pass computes the candidate-aware attention weights over the FULL history
 * (layers.py:66-81: both softmaxes run over all H slots), the scoring kernel evaluates every chunk with those weights and
 * writes its partial pooling state (online softmax + GraphSAGE prefix sum), a merge kernel combines the chunks into the
 * lifetime-weighted score.  If any chunk unit is flagged (remainder bound, fp16 range, operand rows) the exact kernel re-scores
 * the whole set in the same call.  scratch: lime_score_long_scratch_ints(chunked->num_units, imp->num_units) int32; work:
 * lime_score_long_work_floats(num_pairs, H, chunks) floats (attention matrix, partial states). */
int64_t lime_score_long_scratch_ints(int32_t chunked_units, int32_t orig_units);
int64_t lime_score_long_work_floats(int64_t num_pairs, int32_t max_history, int32_t chunks);
int lime_score_impressions_long(const LimeNewsCache *cache, const LimeImpressions *imp, const LimeImpressions *chunked,
                                int32_t chunks, int64_t num_pairs, int32_t num_impressions, int64_t pair_index_base,
                                int32_t prefix_main, int64_t tail_start, int32_t prefix_tail, float *scores, int32_t *scratch,
                                float *work, void *stream);

int lime_score_impressions(const LimeNewsCache *cache, const LimeImpressions *imp,
                           int64_t pair_index_base, int32_t prefix_main, int64_t tail_start,
                           int32_t prefix_tail, float *scores, int32_t *scratch,
                           void *stream);
int     lime_score_configure(int32_t mode, float tolerance);
/* Explain scored pairs: the exact kernel's per-slot terms of every (impression, candidate) pair, for the few pairs a user
 * is shown.  Replaces, per pair, the same reference lines as lime_score_impressions
 *   CandidateAware_ClickedNewsAttention.forward   layers.py:52-93
 *   userEncoders.CROWN.forward tail               userEncoders.py:121,151-171
 *   RemainingLifetimeWeighting.forward            util.py:23-49
 * and writes the score as a sum of one term per history slot plus a bias (DESIGN.md "Explaining a recommendation"):
 *   scores[p]                   the score, the same expression (and, in SCORE_EXACT mode, the same bits) as
 *                               lime_score_impressions;
 *   weight[p]                   w = the remaining-lifetime weight;
 *   bias[p]                     w * (b_l . c + (1/P) sum_{j < P - H} user_node_j . W_l^T c), the part no history slot carries;
 *   alpha[p * H + h]            the candidate-query pooling weight of slot h (userEncoders.py:164, unmasked);
 *   topic_attn[p * H + h]       the candidate-aware weight of slot h (layers.py:81, unmasked);
 *   contrib[p * H + h]          w * (alpha_h x_h . W_r^T c + [h < min(P, H)] x_h . W_l^T c / P),
 * so scores[p] = bias[p] + sum_h contrib[p * H + h] up to fp32 rounding.  P = prefix_main for every pair.  Always runs the
 * exact kernel, whatever lime_score_configure selected.  A unit with unit_count 0 is skipped; the pairs no unit covers are
 * not written.  H in [1, 224], prefix_main in [1, H + user_nodes], every pointer non-null; scratch: lime_score_scratch_ints. */
int     lime_explain_pairs(const LimeNewsCache *cache, const LimeImpressions *imp, int32_t prefix_main, float *scores,
                           float *alpha, float *topic_attn, float *contrib, float *bias, float *weight, int32_t *scratch,
                           void *stream);
/* Candidate-aware attention logits depend on the news only through their (category, subCategory)
 * pair (layers.py:66-70 on the 50-d topic representations), so they are tabulated once per checkpoint:
 *   out[(tc * T + th) * LIME_TOPIC_TAB_LD + head] = exp(Q_head(topic tc) . K_head(topic th) / sqrt(D))   (softmax numerators)
 * topics [T, ldt]: topic representation of every distinct topic (50 used columns);
 * tq [T, ldq]: the [50*10 | 10] candidate-role affine image of the same topics (LIME_CAND_TQ block). */
int     lime_topic_pair_table(const float *topics, int64_t ldt, const float *tq, int64_t ldq, int32_t T,
                              float *out, void *stream);
/* fp32 -> fp16 hi/lo pairs for the tensor-core scoring path: src [rows, lds] holds `blocks` blocks of
 * LIME_D columns; dst [rows, blocks * 2 * LIME_D] fp16 receives per block the hi halves then the lo halves
 * (scale * x = hi + lo to 2^-22; the scoring kernel expects scale = LIME_CAND16_SCALE).  absmax (may be NULL): absmax[row * ldo] = max |x| of the row (inf for NaN). */
int     lime_split_f16_pairs(const float *src, int64_t lds, int64_t rows, int32_t blocks, float scale, void *dst,
                             float *absmax, int64_t ldo, void *stream);
/* Write n freshly built cache rows into a news-vector cache of news_num rows (csrc/cache.cu): source row r = hist [n,
 * LIME_HIST_LD] and cand [n, LIME_CAND_LD] (contiguous, topic ids stamped) goes to destination row dst_rows[r] (int64) of
 * every role, in one pass:
 *   hist_rows [news_num, LIME_HIST_LD] and cand_rows [news_num, LIME_CAND_LD]: copies, max |cand[:, :1200]| (inf for NaN)
 *     stamped into LIME_CAND_ABSMAX;
 *   cand16 [>= news_num, LIME_CAND16_LD] fp16: the hi / lo pairs of lime_split_f16_pairs (scale LIME_CAND16_SCALE, same
 *     arithmetic, bit for bit); the tail of bucket-pair rows after news_num is not touched;
 *   news_meta [news_num, LIME_META_LD]: topic id | gw absmax | w absmax | B1 B2 B3 cb | 0;
 *   hist_vg [news_num, 2*LIME_D]: vc and gw interleaved by 4 dims.
 * The source rows may be the destination rows themselves (dst_rows[r] = r, same memory); otherwise they must not overlap the
 * destination, and dst_rows must not repeat a row (the caller checks).  A destination outside [0, news_num) is skipped: the
 * ids live on the device, so they are not checked here.  Every array 16-byte aligned.  n == 0: no launch. */
int     lime_cache_write_rows(const float *hist, const float *cand, int64_t n, const int64_t *dst_rows, float *hist_rows,
                              float *cand_rows, void *cand16, float *news_meta, float *hist_vg, int64_t news_num, void *stream);
/* Diagnostic: per-phase clock64() totals of the tensor-core scoring kernel since the last call (thread 0 of every CTA;
 * slots listed in score_tc.cu), host buffer of 16 uint64.  Synchronises the device. */
int     lime_score_phase_clocks(uint64_t *out16);
int64_t lime_score_scratch_ints(int32_t num_units);
/* Work-unit capacity (candidates per unit) to build the unit list with for a given H; 0 = unsupported. */
int32_t lime_score_tile_c(int32_t max_history);
/* Dynamic shared memory the exact scoring kernel needs for (H, tile_c); > 232448 means unsupported. */
int64_t lime_score_smem_bytes(int32_t max_history, int32_t tile_c);

/* ---- compute_scores' ranking (util.py:113-123) + evaluate.scoring (evaluate.py:32-89) ---------
 * Per impression i with candidates cand_off[i]..cand_off[i+1]: stable descending rank (ties keep
 * candidate order, -0.0 == 0.0), then AUC / MRR / nDCG@5 / nDCG@10 with y_score = 1/rank in fp64.
 * ranks [P] int32 (may be NULL), metrics [I, 4] fp64.  Impressions without candidates get NaNs
 * and are skipped by lime_metrics_reduce (evaluate.py:44-45).                                     */
int lime_rank_metrics(const float *scores, const uint8_t *labels, const int64_t *cand_off,
                      int64_t num_impressions, int32_t *ranks, double *metrics, void *stream);
/* sums[0..3] = sum over valid impressions of the 4 metrics, sums[4] = number of valid impressions
 * (deterministic fixed-order reduction; the caller divides, or all-reduces across ranks first).  */
int lime_metrics_reduce(const double *metrics, int64_t num_impressions, double *sums, void *stream);

/* ---- top-k news of a pool per user (recommend.top_k; csrc/topk.cu) ---------------------------
 * Top-k of every user's scores over a news pool.
 * scores [users, pool] fp32: row u = user u's scores in PLAN order (position c of the pool plan).
 * pool_index [pool] int32: the caller's index of plan position c (output id and tie-break key).
 * pool_news [pool] int32: cache row of position c (used only for the clicked-history exclusion).
 * exclude [pool] uint8 or NULL: nonzero = never returned (expired news, caller filters).
 * hist_news / hist_mask [users, max_history] or NULL: a position whose pool_news equals a masked-in history
 *   slot of user u is never returned to u (padding slots, mask 0, exclude nothing).
 * Order: descending score; equal scores (-0.0 == +0.0) by ascending pool_index -- the order of
 *   lime_rank_metrics on the pool in the caller's order.  NaN scores are never returned.
 * out_index [users, k] int32 (caller's pool index, -1 past out_count), out_score [users, k] fp32 (-inf past
 *   out_count), out_count [users] int32 = min(k, returnable positions).  1 <= k <= LIME_TOPK_MAX (1024).
 *   A returned -0.0 score reads +0.0.
 * scratch: caller-owned device buffer of lime_pool_topk_scratch_bytes(users, pool, k) bytes (0: may be NULL). */
#define LIME_TOPK_MAX 1024
int64_t lime_pool_topk_scratch_bytes(int32_t users, int64_t pool, int32_t k);
int     lime_pool_topk(const float *scores, int32_t users, int64_t pool, const int32_t *pool_index,
                       const int32_t *pool_news, const uint8_t *exclude, const int32_t *hist_news,
                       const uint8_t *hist_mask, int32_t max_history, int32_t k, int32_t *out_index,
                       float *out_score, int32_t *out_count, void *scratch, void *stream);

/* ---- rank of held-out clicks in the whole pool (recommend.evaluate; csrc/topk.cu) -----------
 * For each user u: the rank of every target among the positions lime_pool_topk could return to u, and ranking
 * metrics of the ranked targets.  scores / pool_index / pool_news / exclude / hist_news / hist_mask / max_history
 * as in lime_pool_topk (pool_news is required only with hist_news).
 * Eligible positions: not marked by exclude, score not NaN, and (with hist_news) news not in u's masked-in history.
 *   They are ordered by lime_pool_topk's key: score descending (-0.0 == +0.0), then ascending pool_index.
 * target_pos [users, targets] int32: pool positions (plan order) of u's held-out clicks; -1 (or any value outside
 *   [0, pool)) = no target.  1 <= targets <= LIME_POOL_RANK_MAX_TARGETS.
 * out_rank [users, targets] int32: 1-based position of the target in u's order, counting every eligible position
 *   (other targets included), so rank r <= k means lime_pool_topk(k) returns it at position r.  0 = unranked: no
 *   target, an ineligible position, or a second or later copy of a position already listed for u.
 * out_ranked [users] int32 = n, the ranked targets; out_eligible [users] int64 = N, the eligible positions.
 * out_metrics [users, 4 + 2 * num_cutoffs] fp64 = auc, mrr, ndcg5, ndcg10, then recall@K, ndcg@K per cutoff K:
 *   auc = (sum (N - r_i) - n(n-1)/2) / (n (N - n)) (integer numerator; NaN when N == n), mrr = mean 1/r_i,
 *   ndcg@K = sum_{r_i <= K} 1/log2(r_i + 1) over the ideal sum_{i <= min(n, K)} 1/log2(i + 1), recall@K =
 *   #{r_i <= K} / n -- the formulas of lime_rank_metrics.  n == 0: an all-NaN row.
 * cutoffs: HOST array of num_cutoffs (<= LIME_POOL_RANK_MAX_CUTOFFS) values >= 1, passed by value into the launch.
 * scratch: caller-owned device buffer of lime_pool_rank_scratch_bytes(users, targets) bytes; zeroed here on `stream`. */
#define LIME_POOL_RANK_MAX_TARGETS 256
#define LIME_POOL_RANK_MAX_CUTOFFS 8
int64_t lime_pool_rank_scratch_bytes(int32_t users, int32_t targets);
int     lime_pool_rank_metrics(const float *scores, int32_t users, int64_t pool, const int32_t *pool_index,
                               const int32_t *pool_news, const uint8_t *exclude, const int32_t *hist_news,
                               const uint8_t *hist_mask, int32_t max_history, const int32_t *target_pos, int32_t targets,
                               const int32_t *cutoffs, int32_t num_cutoffs, int32_t *out_rank, int32_t *out_ranked,
                               int64_t *out_eligible, double *out_metrics, void *scratch, void *stream);


/* ---- training: backward kernels of the same path (trainer.py:131-146 differentiates through them) ----
 * Parameter gradients are ACCUMULATED into caller-zeroed buffers; activation gradients are overwritten. */
/* C (+)= alpha * op(A) . op(B).  a_kmajor: element (i, kk) of op(A) at A[i*lda + kk], else A[kk*lda + i];
 * b_kmajor: element (kk, j) of op(B) at B[j*ldb + kk] (an nn.Linear weight), else B[kk*ldb + j].
 * nn.Linear backward: dX = lime_gemm(dY, 1, W, 0), dW = lime_gemm(dY, 0, X, 0) (split-K over the tokens). */
int lime_gemm(const float *A, int64_t lda, int a_kmajor, const float *B, int64_t ldb, int b_kmajor, float *C,
              int64_t ldc, int64_t m, int n, int64_t k, float alpha, int accumulate, void *stream);
/* bf16 mode of lime_gemm: operands rounded to bf16, tcgen05 tensor cores, fp32 accumulation in TMEM. */
int lime_gemm_bf16(const float *A, int64_t lda, int a_kmajor, const float *B, int64_t ldb, int b_kmajor, float *C,
                   int64_t ldc, int64_t m, int n, int64_t k, float alpha, int accumulate, void *stream);
/* The weight gradient dW = dZ^T . X of an nn.Linear in bf16 mode on bf16 IMAGES of the operands (lime_split_bf16_pairs with
 * lo = NULL): C[m, n] (+)= alpha * sum_{r < k} A[r, i] * B[r, j], A [k, lda] and B [k, ldb] bf16 row-major over the k token
 * rows (lda, ldb multiples of 8, 16-byte aligned).  TMA-fed tcgen05 kernel, both operands MN-major, split-K over the rows
 * with atomicAdd (csrc/gemm_tma.cu).  Replaces lime_gemm_bf16(dY, 0, X, 0) of the round-1 training path. */
int lime_gemm_bf16_tn_tma(const void *A, int64_t lda, const void *B, int64_t ldb, float *C, int64_t ldc, int32_t m,
                          int32_t n, int64_t k, float alpha, int32_t accumulate, void *stream);
/* dx = dy * act'(.) evaluated from the OUTPUT y of the fused activation (1 relu, 2 tanh) */
int lime_act_bwd(const float *dy, int64_t lddy, const float *y, int64_t ldy, float *dx, int64_t lddx,
                 int64_t rows, int cols, int act, void *stream);
/* out[c] += sum_r M[r, c]  (bias gradients) */
int lime_col_sum(const float *M, int64_t ld, int64_t rows, int cols, float *out, void *stream);
/* nn.LayerNorm backward from the layer INPUT x.  bcast_T > 0: dy holds one row per news and row r uses
 * dy[r / bcast_T] / bcast_T (backward of the token mean, newsEncoders.py:317,321). */
int lime_layernorm_bwd(const float *x, int64_t ldx, const float *gamma, const float *dy, int64_t lddy,
                       int bcast_T, float *dx, int64_t lddx, float *dgamma, float *dbeta, int64_t rows, int d,
                       float eps, void *stream);
/* out[r, :d] = table[ids[r], :d]  /  dtable[ids[r], :d] += src[r, :d]  (embedding forward / backward) */
int lime_gather_rows(const float *table, int64_t ldt, int64_t table_rows, const int32_t *ids, int64_t n, int d,
                     float *out, int64_t ldo, void *stream);
int lime_scatter_add_rows(const float *src, int64_t lds, const int32_t *ids, int64_t n, int d, float *dtable,
                          int64_t ldt, int64_t table_rows, void *stream);
/* the same accumulation for large id lists with hot rows (word-embedding gradient): sorted_ids ascending, perm[k] = the row of
 * src that belongs to sorted position k (torch.sort of the ids); runs of equal ids are summed in registers, one 128-bit
 * reduction per run and 32-position chunk.  d <= 512, d / lds / ldt multiples of 4, 16-byte aligned bases. */
int lime_scatter_add_rows_sorted(const float *src, int64_t lds, const int32_t *sorted_ids, const int64_t *perm, int64_t n,
                                 int d, float *dtable, int64_t ldt, int64_t table_rows, void *stream);
/* backward of lime_mha: dctx [n_news*T, d] -> dqkv [n_news*T, 3d] */
int lime_mha_bwd(const float *qkv, const float *dctx, float *dqkv, int64_t n_news, int T, int d, int nhead,
                 float p_drop, uint64_t seed, int64_t news0,
                 void *stream);
/* bf16 mode of lime_mha for the training layout (fp32 qkv / ctx, same dropout mask): S = Q K^T and O = (P M) V on the
 * tensor cores (mma.sync m16n8k16), softmax in fp32 on the accumulator fragments. */
int lime_mha_fwd_bf16(const float *qkv, float *ctx, int64_t n_news, int T, int d, int nhead, float p_drop, uint64_t seed,
                      int64_t news0, void *stream);
/* fp32x3 mode of lime_mha (Stage A, same arguments and layouts): q, k, v and the softmax weights as fp16 hi / lo pairs
 * (22 significant bits), each product three mma.sync m16n8k16 passes with fp32 accumulation -- fp32-level accuracy
 * on the tensor cores; replaces the FFMA core of newsEncoders.py:244-247's nn.MultiheadAttention in that mode.
 * ctx_hi / ctx_lo != NULL: the context is written as the fp16 pair out_scale * ctx = hi + lo, each [rows, ld16] with columns
 * d..ld16-1 zero (the A operand of the out_proj lime_linear_x3_tma: no fp32 copy, no lime_split_bf16_pairs pass); ctx is
 * then not written and may be NULL. */
int lime_mha_x3(const float *qkv, float *ctx, void *ctx_hi, void *ctx_lo, int32_t ld16, float out_scale, int64_t n_news, int T,
                int d, int nhead, float p_drop, uint64_t seed, int64_t news0, void *stream);
/* bf16 mode of lime_mha_bwd: q, k, v, dO rounded to bf16, every product of the backward on the tensor cores (mma.sync
 * m16n8k16, fp32 accumulation), softmax statistics in fp32; same arguments and dropout mask. */
int lime_mha_bwd_bf16(const float *qkv, const float *dctx, float *dqkv, int64_t n_news, int T, int d, int nhead,
                      float p_drop, uint64_t seed, int64_t news0, void *stream);
/* backward of lime_intent_pool: dout [n, D] -> dpre, de [n, k, D], dw2 [D] (accumulated) */
int lime_intent_pool_bwd(const float *pre, const float *e, const float *w2, const float *dout, int64_t lddo,
                         float *dpre, float *de, float *dw2, int64_t n, int k, int D, void *stream);
/* backward of lime_content_fuse w.r.t. title / body (the category slices of dcontent are scattered by the
 * caller with lime_scatter_add_rows) */
int lime_content_fuse_bwd(const float *title, const float *body, const float *dcontent, int64_t ldc, int64_t n,
                          int D, float *dtitle, float *dbody, void *stream);
/* inverted dropout, stateless: y = x * keep(seed, element index) / (1 - p); the backward is the same call
 * on the gradient with the same seed */
int lime_dropout(const float *x, int64_t ldx, float *y, int64_t ldy, int64_t rows, int cols, float p,
                 uint64_t seed, void *stream);
/* fused forms with the SAME masks: y = x * m(seed) [* m(seed2) if two_masks] [+ res if res != NULL] (the post-LN residual
 * branches dropout(sublayer(x)) + x of nn.TransformerEncoderLayer, newsEncoders.py:244-247, in one pass; two masks = the
 * backward of lime_embed_pe_dropout).  cols and leading dimensions multiples of 4, 16-byte aligned bases. */
int lime_dropout_fused(const float *x, int64_t ldx, const float *res, int64_t ldr, float *y, int64_t ldy, int64_t rows,
                       int cols, float p, uint64_t seed, uint64_t seed2, int two_masks, void *stream);
/* training-mode embedding path in one pass (newsEncoders.py:311-315, :828): out[r, c] = m_x * (m_w * E[ids[r], c] + pe[r % T, c]),
 * m_w / m_x the dropout masks of (seed_w, r d + c) / (seed_x, r d + c) -- what lime_gather_rows, lime_dropout, the positional add
 * and a second lime_dropout compute.  E [vocab, d] and out [rows, d] contiguous, d a multiple of 4. */
int lime_embed_pe_dropout(const float *E, int64_t vocab, const int32_t *ids, int64_t rows, int T, int d, const float *pe,
                          float p, uint64_t seed_w, uint64_t seed_x, float *out, void *stream);

/* ---- training: CROWN user encoder + click score, N candidates per sample (userEncoders.py:101-175,
 * layers.py:52-93, util.py:23-49).  Dense layers are lime_linear / lime_gemm; these are the pieces between. */
/* a[b, h] of CandidateAware_ClickedNewsAttention from Qp = query_proj(t_c) [B,N,400], Kp = key_proj(t_h)
 * [B,H,400], mask [B,H] (layers.py:66-81) and its backward.  p_drop: dropout on the per-head attention weights
 * (layers.py:36,74, nn.Dropout(0.2) in training; 0 in eval), stateless mask of (seed, sample, index) -- the backward
 * call must pass the forward's p_drop and seed. */
int lime_ca_attention_fwd(const float *Qp, const float *Kp, const uint8_t *mask, int32_t B, int32_t N, int32_t H,
                          float p_drop, uint64_t seed, float *a, void *stream);
int lime_ca_attention_bwd(const float *Qp, const float *Kp, const uint8_t *mask, int32_t B, int32_t N, int32_t H,
                          float p_drop, uint64_t seed, const float *da, float *dQp, float *dKp, void *stream);
/* wc = a * v per row (layers.py:84) */
int lime_row_scale_fwd(const float *v, const float *a, int64_t rows, int d, float *out, void *stream);
int lime_row_scale_bwd(const float *v, const float *a, const float *dwc, int64_t rows, int d, float *dv, float *da,
                       void *stream);
/* o = sigmoid(z) * wc + (1 - sigmoid(z)) * v (layers.py:87-88), elementwise over `total` values */
int lime_gate_mix_fwd(const float *z, const float *wc, const float *v, int64_t total, float *o, void *stream);
int lime_gate_mix_bwd(const float *z, const float *wc, const float *v, const float *dout, int64_t total, float *dz,
                      float *dwc, float *dv, void *stream);
/* GraphSAGE mean over node indices 0..P-1 of [x_b (H rows) ; user_node rows] (userEncoders.py:91-98,121,153) */
int lime_sage_mean_fwd(const float *x, const float *un, int32_t B, int32_t H, int32_t P, int32_t un_rows, float *m,
                       void *stream);
int lime_sage_mean_bwd(const float *dm, int32_t B, int32_t H, int32_t P, int32_t un_rows, float *dx, float *dun,
                       void *stream);
/* g[b,h] = r[b,h] + l[b]  /  dl[b] = sum_h dg[b,h] */
int lime_add_row_bcast(const float *r, const float *l, int64_t rows, int32_t H, int d, float *g, void *stream);
int lime_sum_over_h(const float *dg, int32_t B, int32_t H, int d, float *dl, void *stream);
/* candidate-query pooling (userEncoders.py:158-171): Kg = K(g) [B,H,400], q = Q(c) [B,N,400], g [B,H,400]
 * -> u [B,N,400], alpha [B,N,H] (saved for the backward) */
int lime_pool_fwd(const float *Kg, const float *q, const float *g, int32_t B, int32_t N, int32_t H, float *u,
                  float *alpha, void *stream);
int lime_pool_bwd(const float *Kg, const float *q, const float *g, const float *alpha, const float *du, int32_t B,
                  int32_t N, int32_t H, float *dKg, float *dq, float *dg, void *stream);
/* scores[r] = (u[r] . c[r]) * w(remaining[r]) (util.py:23-49); w is returned for the backward */
int lime_click_score_fwd(const float *u, const float *c, const float *remaining, int64_t rows, float alpha,
                         float beta, int32_t use_weighting, int32_t use_expired_penalty, float *scores, float *w,
                         void *stream);
int lime_click_score_bwd(const float *u, const float *c, const float *w, const float *dscores, int64_t rows,
                         float *du, float *dc, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* LIME_B200_H_ */
