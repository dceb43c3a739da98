"""Training-mode forward of the drop-in model (reference model.py:151-187 with N = 1 + M candidates per
sample, trainer.py:131-146): the same math as the eval path, composed from differentiable ops whose
forward and backward are liblime_b200.so kernels (autograd.py).  No news-vector cache here: weights
change every step, so every news of the mini-batch is encoded (B * (H + N) encodes, as the reference).

Dropout: the reference drops activations with torch's RNG, whose streams cannot be reproduced; this path
applies inverted dropout at the SAME sites with its own stateless counter-based generator (the backward
re-evaluates the forward's mask): word embeddings, after the positional encoding, inside
nn.TransformerEncoderLayer (attention weights, after out_proj, after the FFN activation, after linear2),
category embeddings, the fixed p = 0.2 on the candidate-aware attention weights (layers.py:36,74) and the
user-node rows.  Gradient parity is tested with every p = 0 (SURVEY.md section 7, tests/test_gpu_training.py)
and with every site live, against the oracle under the same masks (tests/test_gpu_training_parity.py).
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from . import autograd as A
from . import ops

RELU, TANH = ops.ACT_RELU, ops.ACT_TANH


def _branch(base, ids, T, transformer, pos_encoder, heads, p, seed):
    """One transformer branch (title or body): int32 ids [n, T] -> mean-pooled features [n, 300].
    Dropout sites as the reference places them (inverted dropout, stateless masks): word embeddings
    (newsEncoders.py:311-312), after the positional encoding (:828), and inside nn.TransformerEncoderLayer
    (:244-247, post-LN): attention weights, after out_proj, after the FFN activation, after linear2."""
    n = ids.shape[0]
    l = transformer.layers[0]
    d = base.word_embedding.weight.shape[1]
    pe = pos_encoder.pe.reshape(-1, d)
    if p > 0 and d % 4 == 0 and base.word_embedding.weight.is_contiguous():
        # dropout(word embeddings, seed) + pe, dropout(., seed + 1): one kernel with the two masks of the unfused form below
        x0 = A.EmbedPEDropout.apply(base.word_embedding.weight, ids.reshape(-1).contiguous(), T, pe.contiguous(), p, seed, seed + 1)
    elif p > 0:
        w = A.dropout(A.Gather.apply(base.word_embedding.weight, ids.reshape(-1).contiguous()), p, seed)
        x0 = A.dropout(w + pe[:T].repeat(n, 1), p, seed + 1)
    else:
        x0 = A.EmbedPE.apply(base.word_embedding.weight, ids.reshape(-1).contiguous(), T, pe)
    qkv = A.linear(x0, l.self_attn.in_proj_weight, l.self_attn.in_proj_bias)
    ctx = A.MHA.apply(qkv, n, T, d, heads, p, seed + 2)
    if p > 0:
        y = A.dropout_add(A.linear(ctx, l.self_attn.out_proj.weight, l.self_attn.out_proj.bias), x0, p, seed + 3)
    else:
        y = A.linear(ctx, l.self_attn.out_proj.weight, l.self_attn.out_proj.bias, residual=x0)
    x1 = A.LayerNorm.apply(y, l.norm1.weight, l.norm1.bias, l.norm1.eps)
    hf = A.dropout(A.linear(x1, l.linear1.weight, l.linear1.bias, act=RELU), p, seed + 4)
    if p > 0:
        y2 = A.dropout_add(A.linear(hf, l.linear2.weight, l.linear2.bias), x1, p, seed + 5)
    else:
        y2 = A.linear(hf, l.linear2.weight, l.linear2.bias, residual=x1)
    return A.LayerNormMeanPool.apply(y2, l.norm2.weight, l.norm2.bias, n, T, l.norm2.eps)


def topic_representation(owner, category, subCategory):
    """category_affine(category_embedding(c) || subCategory_embedding(s)) -> [n, 50]
    (newsEncoders.py:340-342 with CROWN's tables; userEncoders.py:103-105,115-117 with LIME's)."""
    ce = A.Gather.apply(owner.category_embedding.weight, category)
    se = A.Gather.apply(owner.subCategory_embedding.weight, subCategory)
    return A.linear(torch.cat([ce, se], dim=1), owner.category_affine.weight, owner.category_affine.bias)


def encode_news(lime, title_text, body_text, category, subCategory, freshness, lifetime, seed=0):
    """LIME(CROWN) news encoder, training mode, flat over news:
    int32 [n,32], [n,128], [n], [n], fp32 seconds [n], [n] -> fp32 [n, 400] with an autograd graph."""
    base, cfg = lime.base_news_encoder, lime.config
    p = float(cfg.dropout_rate) if lime.training else 0.0
    n = title_text.shape[0]
    heads = cfg.head_num
    ft = _branch(base, title_text, title_text.shape[1], base.title_transformer, base.title_pos_encoder, heads, p, seed + 11)
    fb = _branch(base, body_text, body_text.shape[1], base.body_transformer, base.body_pos_encoder, heads, p, seed + 23)
    t = topic_representation(base, category, subCategory)                                   # [n, 50]
    k = len(base.intent_layers)
    W = F.pad(torch.cat([lin.weight for lin in base.intent_layers], dim=0), (0, 2))         # [k*400, 352]
    b = torch.cat([lin.bias for lin in base.intent_layers], dim=0)
    pad = torch.zeros(n, 2, dtype=torch.float32, device=ft.device)
    pooled = []
    for feat, att in ((ft, base.title_intent_attention), (fb, base.body_intent_attention)):
        e = A.linear(torch.cat([feat, t, pad], dim=1), W, b, act=RELU).view(n * k, -1)      # [n*k, 400]
        pre = A.linear(e, att.affine1.weight, att.affine1.bias)
        pooled.append(A.IntentPool.apply(pre, e, att.affine2.weight.reshape(-1), n, k))
    content = A.ContentFuse.apply(pooled[0], pooled[1], base.category_embedding.weight,
                                  base.subCategory_embedding.weight, category, subCategory, p, seed + 37)
    fe = lime.freshness_encoder
    nb = fe.num_buckets
    pairs = A.BucketPairs.apply(fe.freshness_embedding.weight, fe.lifetime_embedding.weight)
    table = A.linear(pairs, fe.dense.weight, fe.dense.bias, act=TANH)                       # [nb*nb, 900]
    idx = (ops.bucketize(freshness.reshape(-1).float().contiguous(), nb) * nb
           + ops.bucketize(lifetime.reshape(-1).float().contiguous(), nb)).to(torch.int32)
    fresh = A.Gather.apply(table, idx)
    cd = content.shape[1]
    pw = lime.project.weight
    return A.linear(fresh, pw[:, cd:], None, residual=A.linear(content, pw[:, :cd], lime.project.bias))


def user_representation(ue, hist_vec, cand_vec, hist_cat, hist_sub, cand_cat, cand_sub, hist_mask, B, H, N, seed=0):
    """userEncoders.CROWN.forward after the history encode (userEncoders.py:103-105,114-175):
    hist_vec [B*H,400], cand_vec [B*N,400] (LIME vectors), int32 category ids flat, mask uint8 [B,H]
    -> user representation [B*N, 400], every step a liblime_b200 kernel with its backward."""
    lime, cfg = ue.news_encoder, ue.config
    ca = ue.candidate_aware_attn
    sage = ue.graph_sage.convs[0]
    p = float(cfg.dropout_rate) if ue.training else 0.0
    # topic representations from LIME's frozen tables + category_affine (userEncoders.py:103-105,115-117)
    pad_h = torch.zeros(B * H, 2, dtype=torch.float32, device=hist_vec.device)
    pad_c = torch.zeros(B * N, 2, dtype=torch.float32, device=hist_vec.device)
    th = torch.cat([topic_representation(lime, hist_cat, hist_sub), pad_h], dim=1)            # [B*H, 52]
    tc = torch.cat([topic_representation(lime, cand_cat, cand_sub), pad_c], dim=1)            # [B*N, 52]
    Qp = A.linear(tc, F.pad(ca.query_proj.weight, (0, 2)), ca.query_proj.bias)                # layers.py:66
    Kp = A.linear(th, F.pad(ca.key_proj.weight, (0, 2)), ca.key_proj.bias)                    # layers.py:67
    a = A.CAAttention.apply(Qp, Kp, hist_mask, B, N, H, float(ca.dropout.p) if ue.training else 0.0, seed + 61)   # [B*H]; nn.Dropout(0.2), layers.py:36,74
    wc = A.RowScale.apply(hist_vec, a)                                                         # layers.py:84
    z = A.linear(wc, ca.gate_proj.weight, ca.gate_proj.bias)
    o = A.GateMix.apply(z, wc, hist_vec)                                                       # layers.py:87-88
    x = A.LayerNorm.apply(o, ca.layernorm.weight, ca.layernorm.bias, ca.layernorm.eps)
    # GraphSAGE over [x ; dropout(user_node_embedding)], sources = runtime batch (userEncoders.py:91-98,121,151-157)
    un = A.dropout(ue.user_node_embedding, p, seed + 51)
    m = A.SageMean.apply(x, un, B, H, B)
    g = A.AddRowBroadcast.apply(A.linear(x, sage.lin_r.weight, None), A.linear(m, sage.lin_l.weight, sage.lin_l.bias), H)
    # candidate-query pooling (userEncoders.py:158-171)
    Kg = A.linear(g, ue.K.weight, None)
    q = A.linear(cand_vec, ue.Q.weight, ue.Q.bias)
    return A.Pool.apply(Kg, q, g, B, N, H)


def click_scores(rw, u, cand_vec, remaining, B, N):
    """RemainingLifetimeWeighting.forward (util.py:23-49): u, cand_vec [B*N, 400], remaining [B*N] -> [B, N]."""
    s = A.ClickScore.apply(u, cand_vec, remaining.reshape(-1).float().contiguous(), rw.alpha, rw.beta,
                           rw.use_remaining_lifetime_weighting, rw.use_expired_penalty)
    return s.view(B, N)


def user_scores(model, hist_vec, cand_vec, hist_cat, hist_sub, cand_cat, cand_sub, hist_mask, remaining, B, H, N, seed=0):
    """CROWN user encoder + lifetime-weighted click score, training layout -> logits [B, N]
    (userEncoders.py:101-175, util.py:23-49)."""
    u = user_representation(model.user_encoder, hist_vec, cand_vec, hist_cat, hist_sub, cand_cat, cand_sub, hist_mask,
                            B, H, N, seed)
    return click_scores(model.remaining_lifetime_weighting, u, cand_vec, remaining, B, N)


def model_forward(model, user_category, user_subCategory, user_title_text, user_content_text, user_freshness,
                  user_lifetime, user_history_mask, news_category, news_subCategory, news_title_text,
                  news_content_text, news_freshness, news_lifetime, remaining_lifetime, seed=0):
    """Training-mode Model.forward (model.py:151-187): candidate tensors carry the news dim N."""
    B, H = user_category.shape
    N = news_category.shape[1]
    i32 = torch.int32
    flat = lambda t, w: t.reshape(-1, w).to(i32).contiguous()
    title = torch.cat([flat(user_title_text, user_title_text.shape[-1]), flat(news_title_text, news_title_text.shape[-1])])
    body = torch.cat([flat(user_content_text, user_content_text.shape[-1]), flat(news_content_text, news_content_text.shape[-1])])
    cat = torch.cat([user_category.reshape(-1), news_category.reshape(-1)]).to(i32).contiguous()
    sub = torch.cat([user_subCategory.reshape(-1), news_subCategory.reshape(-1)]).to(i32).contiguous()
    fresh = torch.cat([user_freshness.reshape(-1), news_freshness.reshape(-1)]).float().contiguous()
    life = torch.cat([user_lifetime.reshape(-1), news_lifetime.reshape(-1)]).float().contiguous()
    vec = encode_news(model.news_encoder, title, body, cat, sub, fresh, life, seed)            # [B*H + B*N, 400]
    hist_vec, cand_vec = vec[:B * H], vec[B * H:]
    return user_scores(model, hist_vec, cand_vec, cat[:B * H], sub[:B * H], cat[B * H:], sub[B * H:],
                       user_history_mask.to(torch.uint8).contiguous(), remaining_lifetime, B, H, N, seed)
