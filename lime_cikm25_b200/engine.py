"""Host-side driver of the B200 path: weight preparation, news-vector cache build (Stage A) and
impression scoring (Stage B).  All arithmetic is done by liblime_b200.so through ``ops``; torch
supplies device buffers, views/copies and the current stream.

Layout of the per-news cache in HBM (fp32; DESIGN.md "HBM layout"):

  hist_rows [news, 852]   vc = W_c content            (0..399)   LIME projection, content half, no bias
                          gw = -log2(e) W_g vc          (400..799) gate pre-activation of the history role
                          t  = topic representation     (800..851) LIME's frozen tables, padded 50->52
  cand_rows [news, 1720]  w1 = gamma*P vc/20 | w2 = gamma*W_r^T vc | w3 = gamma*W_l^T vc   (0..1199)
                          7 scalars (1200..1206), tq 50x10 (1208..1707), qb 10 (1708..1717)
  hist_tab  [nb*nb, 800]  the same two history vectors for T[bf,bl] = W_f tanh(dense(E_f|E_l)) + b
  cand_tab  [nb*nb, 1208] the same candidate block for T[bf,bl] (+ the constants coming from Q.bias)
  cand16    [news + R*nb*nb, 2400]  fp16 [hi | lo][w1 w2 w3][400]: cand_rows as hi/lo pairs (x = hi + lo to 2^-22),
                          the M operand of the tensor-core scoring kernel, streamed by cp.async without touching
                          registers; the tail holds R = 32 copies of the same for cand_tab (ctab16): every CTA of the
                          scoring kernel reads its own copy of the hot bucket-pair rows (hist_tab likewise)

A LIME news vector is v(news, bf, bl) = vc[news] + T[bf, bl]; everything the scoring kernel needs is
linear in v, so it is cached as a per-news part plus a per-bucket-pair part.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from . import _lib, ops
from ._lib import LimeImpressions, LimeNewsCache, check

D = 400
HIST_LD, CAND_LD, HTAB_LD, CTAB_LD = 852, 1720, 800, 1208
HIST_GW, HIST_T, HIST_TOPIC_ID, HIST_GW_ABSMAX = 400, 800, 850, 851
CAND_SCAL, CAND_TQ, CAND_NFOLD, CAND_TOPIC_ID, CAND_ABSMAX = 1200, 1208, 1207, 1718, 1207
F16_SAFE = 32768.0 / ops.CAND16_SCALE      # |w| beyond this leaves the fp16 operand range after scaling
TOPIC_TAB_LD, MAX_TOPICS, TC_MAX_HISTORY = 12, 1024, 56
TC_TRIPLES = 40         # operand-row triples of a tensor-core work unit: candidates + distinct bucket pairs
TAB_REPLICAS = 32      # copies of the bucket-pair tables read by the tensor-core kernel (spreads the hot rows over L2 slices)
TOPIC, TOPIC_LD, HEADS = 50, 52, 10
LOG2E = 1.4426950408889634


def interleave_vg(rows):
    """[n, >= 800] fp32 (v | g) -> [n, 800] with v and g interleaved in groups of 4 dims (v0..3 g0..3 v4..7 ...):
    the tensor-core scoring kernel fetches both operands of 4 dims with one 256-bit load (layout copy: plumbing)."""
    n = rows.shape[0]
    return torch.stack([rows[:, :D].reshape(n, D // 4, 4), rows[:, D:2 * D].reshape(n, D // 4, 4)], dim=2).reshape(n, 2 * D).contiguous()


def _fingerprint(params):
    return tuple((p.data_ptr(), p._version) for p in params)


def _check_geometry(cfg):
    """The kernels are specialised for the LIME-CROWN-CROWN geometry of config.py's defaults."""
    want = dict(word_embedding_dim=300, head_num=10, feedforward_dim=512, intent_embedding_dim=400,
                intent_num=3, attention_dim=400, category_embedding_dim=50, subCategory_embedding_dim=50,
                lime_output_dim=400, fusion_method="concat", num_layers=1,
                use_candidate_ware_clicked_news_attention=True, use_residual_connection=True,
                click_predictor="dot_product", alpha=0.0)      # alpha != 0: the category-predictor auxiliary loss is not built
    for k, v in want.items():
        if getattr(cfg, k) != v:
            raise NotImplementedError("lime_cikm25_b200 supports %s=%r only (got %r)" % (k, v, getattr(cfg, k)))
    if cfg.max_title_length != 32 or cfg.max_abstract_length != 128:
        raise NotImplementedError("title/body lengths must be 32/128 (config.py:144-163 forces them)")


class NewsEncoderEngine:
    """Stage A: LIME(CROWN) news encoder, eval mode (newsEncoders.py:140-161, 302-373)."""

    def __init__(self, lime_module, cfg):
        _check_geometry(cfg)
        self.m = lime_module
        self.cfg = cfg
        self._prep = None
        self._fp = None
        self.bf16 = False        # "bf16 mode": bf16 activations, the 4 transformer GEMMs by TMA + tcgen05 (lime_linear_bf16_tma)
        self.x3 = False          # "fp32x3 mode" (opt-in; default = the fp32 FFMA kernels, the strict-parity mode): fp32 residual stream, every dense layer on the tensor cores over fp16 hi / lo pairs
        self.x3_mha = True       # fp32x3 mode: attention core on the tensor cores too (lime_mha_x3, fp16 hi / lo pairs); False = the FFMA core
        self.x3_small = True     # tensor-core modes: intent layers, intent-attention affine and the content projection as fp32x3 passes (False = FFMA lime_linear)

    # -- weights -----------------------------------------------------------------------------------
    def _params(self):
        return [p for p in self.m.parameters()] + [b for b in self.m.buffers()]

    def prepare(self):
        fp = _fingerprint(self._params())
        if self._prep is not None and fp == self._fp:
            return self._prep
        m, base = self.m, self.m.base_news_encoder
        dev = base.word_embedding.weight.device
        if dev.type != "cuda":
            raise _lib.LimeError("model parameters must live on a CUDA device (no CPU fallback)")
        f32 = dict(dtype=torch.float32, device=dev)
        P = {}
        # intent layers: one [k*400, 352] weight (K padded 350 -> 352) so the 3 FCs are a single GEMM
        k = len(base.intent_layers)
        W = torch.zeros(k * 400, 352, **f32)
        b = torch.empty(k * 400, **f32)
        for i, lin in enumerate(base.intent_layers):
            W[i * 400:(i + 1) * 400, :350].copy_(lin.weight.detach())
            b[i * 400:(i + 1) * 400].copy_(lin.bias.detach())
        P["intent_w"], P["intent_b"] = W, b
        # tensor-core modes: the intent layers, their attention's first affine and the content half of LIME.project as
        # fp32x3 passes too (fp16 pairs 2^10 w = hi + lo, K padded to a multiple of 64)
        P["intent_w_hi"], P["intent_w_lo"] = ops.split16(W, scale=ops.X3_W_SCALE)
        for name, att in (("title", base.title_intent_attention), ("body", base.body_intent_attention)):
            P[name + "_a1_hi"], P[name + "_a1_lo"] = ops.split16(att.affine1.weight.detach(), scale=ops.X3_W_SCALE)

        def tr(t):
            l = t.layers[0]
            return dict(in_w=l.self_attn.in_proj_weight.detach(), in_b=l.self_attn.in_proj_bias.detach(),
                        out_w=l.self_attn.out_proj.weight.detach(), out_b=l.self_attn.out_proj.bias.detach(),
                        l1_w=l.linear1.weight.detach(), l1_b=l.linear1.bias.detach(),
                        l2_w=l.linear2.weight.detach(), l2_b=l.linear2.bias.detach(),
                        n1_w=l.norm1.weight.detach(), n1_b=l.norm1.bias.detach(),
                        n2_w=l.norm2.weight.detach(), n2_b=l.norm2.bias.detach(),
                        eps1=l.norm1.eps, eps2=l.norm2.eps)
        P["title"], P["body"] = tr(base.title_transformer), tr(base.body_transformer)

        def pad16(w):        # [n, k] fp32 -> bf16 [n, k padded to a multiple of 64 with zeros]: operand of lime_linear_bf16_tma
            n_, k_ = w.shape
            o = torch.zeros(n_, (k_ + 63) // 64 * 64, dtype=torch.bfloat16, device=dev)
            o[:, :k_].copy_(w)
            return o
        heads = int(self.cfg.head_num)
        hd = 300 // heads

        def head_pad(t):     # in_proj rows q | k | v, each [heads * hd, ...] -> heads slices of 32 rows (zero rows after the hd real ones)
            o = torch.zeros((3, heads, 32) + tuple(t.shape[1:]), dtype=t.dtype, device=dev)
            o[:, :, :hd] = t.reshape((3, heads, hd) + tuple(t.shape[1:]))
            return o.reshape((3 * heads * 32,) + tuple(t.shape[1:]))
        for br in (P["title"], P["body"]):
            for name in ("out_w", "l1_w", "l2_w"):
                br[name + "16"] = pad16(br[name])
            br["in_w16"] = pad16(head_pad(br["in_w"]))          # head-padded q | k | v: the layout lime_mha_bf16 reads
            br["in_b_hp"] = head_pad(br["in_b"])
            for name in ("in_w", "out_w", "l1_w", "l2_w"):        # fp16 pairs 2^10 w = hi + lo for the fp32x3 mode
                br[name + "_hi"], br[name + "_lo"] = ops.split16(br[name], scale=ops.X3_W_SCALE)
        P["title_pe"] = base.title_pos_encoder.pe.detach().reshape(-1, 300).contiguous()
        P["body_pe"] = base.body_pos_encoder.pe.detach().reshape(-1, 300).contiguous()
        pw = m.project.weight.detach()                    # [400, 1800] = [W_c | W_f]
        P["Wc"], P["Wf"], P["proj_b"] = pw[:, :900], pw[:, 900:], m.project.bias.detach()
        P["Wc_hi"], P["Wc_lo"] = ops.split16(P["Wc"], scale=ops.X3_W_SCALE)
        self._prep, self._fp = P, fp
        return P

    # -- one transformer branch (title or body) ----------------------------------------------------
    def _branch(self, ids, T, W, pe, feat):
        base = self.m.base_news_encoder
        n = ids.shape[0]
        rows = n * T
        dev = ids.device
        E = base.word_embedding.weight.detach()
        x0 = torch.empty(rows, 300, dtype=torch.float32, device=dev)
        ops.embed_pe(E, ids, T, pe, x0)
        qkv = ops.linear(x0, W["in_w"], W["in_b"], bf16=self.bf16)
        ctx = torch.empty(rows, 300, dtype=torch.float32, device=dev)
        ops.mha(qkv, ctx, n, T, 300, self.cfg.head_num)
        del qkv
        y = ops.linear(ctx, W["out_w"], W["out_b"], residual=x0, bf16=self.bf16)
        x1 = ops.layernorm(y, W["n1_w"], W["n1_b"], out=ctx, eps=W["eps1"])       # reuse ctx
        hf = ops.linear(x1, W["l1_w"], W["l1_b"], act=ops.ACT_RELU, bf16=self.bf16)
        y2 = ops.linear(hf, W["l2_w"], W["l2_b"], residual=x1, out=y, bf16=self.bf16)
        ops.layernorm_meanpool(y2, W["n2_w"], W["n2_b"], feat, n, T, eps=W["eps2"])

    def _branch_bf16(self, ids, T, W, pe, feat):
        """The same branch in bf16 mode: bf16 activations feed TMA + tcgen05 GEMMs (lime_linear_bf16_tma); the residual
        stream and both LayerNorm inputs stay fp32."""
        base = self.m.base_news_encoder
        n = ids.shape[0]
        rows = n * T
        dev = ids.device
        E = base.word_embedding.weight.detach()
        kp = W["in_w16"].shape[1]                                                   # 300 -> 320
        x0 = torch.empty(rows, 300, dtype=torch.float32, device=dev)
        x0b = torch.empty(rows, kp, dtype=torch.bfloat16, device=dev)
        ops.embed_pe_bf16(E, ids, T, pe, x0, x0b)
        qkv = ops.linear_tma(x0b, W["in_w16"], W["in_b_hp"])                        # bf16 [rows, 960], head-padded q | k | v
        ctxb = torch.empty(rows, kp, dtype=torch.bfloat16, device=dev)
        ops.mha_bf16(qkv, ctxb, n, T, 300, self.cfg.head_num)
        del qkv
        y = ops.linear_tma(ctxb, W["out_w16"], W["out_b"], residual=x0, out_bf16=False)
        x1, x1b = ops.layernorm_bf16(y, W["n1_w"], W["n1_b"], x0, x0b, eps=W["eps1"])      # reuse x0 / x0b
        hf = ops.linear_tma(x1b, W["l1_w16"], W["l1_b"], act=ops.ACT_RELU)           # bf16 [rows, 512]
        y2 = ops.linear_tma(hf, W["l2_w16"], W["l2_b"], residual=x1, out=y)
        ops.layernorm_meanpool(y2, W["n2_w"], W["n2_b"], feat, n, T, eps=W["eps2"])

    def _branch_x3(self, ids, T, W, pe, feat):
        """The same branch in the fp32x3 mode: every dense layer on the tensor cores over fp16 hi / lo operand pairs (ops.linear_x3,
        2^-21 relative per product: fp32-level accuracy), attention on mma.sync hi / lo pairs; the residual stream stays fp32 and
        every producer (embedding, attention, LayerNorm, FFN-1) writes the next layer's operand pair itself."""
        base = self.m.base_news_encoder
        n = ids.shape[0]
        rows = n * T
        dev = ids.device
        E = base.word_embedding.weight.detach()
        x0 = torch.empty(rows, 300, dtype=torch.float32, device=dev)
        sa, al = ops.X3_ACT_SCALE, 1.0 / (ops.X3_ACT_SCALE * ops.X3_W_SCALE)
        xh, xl = ops.embed_pe_pairs(E, ids.reshape(-1), T, pe, x0, sa)        # fp32 residual stream + the in_proj operand pair
        qkv = ops.linear_x3(xh, xl, W["in_w_hi"], W["in_w_lo"], W["in_b"], alpha=al)
        del xh, xl
        ctx = torch.empty(rows, 300, dtype=torch.float32, device=dev)       # (re-used below as the LayerNorm output)
        if self.x3_mha:
            ch, cl = ops.mha_x3_pairs(qkv, n, T, 300, self.cfg.head_num, sa)   # the context leaves as out_proj's operand pair
        else:
            ops.mha(qkv, ctx, n, T, 300, self.cfg.head_num)
            ch, cl = ops.split16(ctx, scale=sa)
        del qkv
        y = ops.linear_x3(ch, cl, W["out_w_hi"], W["out_w_lo"], W["out_b"], residual=x0, alpha=al)
        del ch, cl
        x1 = ctx                                                                 # reuse ctx
        xh, xl = ops.layernorm_pairs(y, W["n1_w"], W["n1_b"], x1, sa, eps=W["eps1"])   # fp32 residual stream + the FFN-1 operand pair
        if ops.X3_FUSED:            # the FFN hidden layer leaves its GEMM as FFN-2's operand pair
            hh, hl = ops.linear_x3_pairs(xh, xl, W["l1_w_hi"], W["l1_w_lo"], W["l1_b"], act=ops.ACT_RELU, alpha=al, out_scale=sa)
            del xh, xl
        else:
            hf = ops.linear_x3(xh, xl, W["l1_w_hi"], W["l1_w_lo"], W["l1_b"], act=ops.ACT_RELU, alpha=al)
            del xh, xl
            hh, hl = ops.split16(hf, scale=sa)
            del hf
        y2 = ops.linear_x3(hh, hl, W["l2_w_hi"], W["l2_w_lo"], W["l2_b"], residual=x1, out=y, alpha=al)
        ops.layernorm_meanpool(y2, W["n2_w"], W["n2_b"], feat, n, T, eps=W["eps2"])

    def encode_content(self, title_text, body_text, category, subCategory):
        """newsEncoders.CROWN.forward, flat over news: int32 [n,32], [n,128], [n], [n] -> fp32 [n,900]."""
        P = self.prepare()
        base = self.m.base_news_encoder
        n = title_text.shape[0]
        dev = title_text.device
        f32 = dict(dtype=torch.float32, device=dev)
        feat_t = torch.empty(n, 352, **f32)
        feat_b = torch.empty(n, 352, **f32)
        branch = self._branch_bf16 if self.bf16 else (self._branch_x3 if self.x3 else self._branch)
        branch(title_text, 32, P["title"], P["title_pe"], feat_t)
        branch(body_text, 128, P["body"], P["body_pe"], feat_b)
        # category-aware intent disentanglement (:340-356): topic from CROWN's own tables
        for feat in (feat_t, feat_b):
            ops.topic_rep(base.category_embedding.weight.detach(), base.subCategory_embedding.weight.detach(),
                          base.category_affine.weight.detach(), base.category_affine.bias.detach(),
                          category, subCategory, feat[:, 300:], TOPIC_LD)
        k = len(base.intent_layers)
        pooled = []
        tc_mode = (self.bf16 or self.x3) and self.x3_small
        sa, al = ops.X3_ACT_SCALE, 1.0 / (ops.X3_ACT_SCALE * ops.X3_W_SCALE)
        for feat, att, name in ((feat_t, base.title_intent_attention, "title"), (feat_b, base.body_intent_attention, "body")):
            if tc_mode:
                fh, fl = ops.split16(feat, scale=sa)
                e = ops.linear_x3(fh, fl, P["intent_w_hi"], P["intent_w_lo"], P["intent_b"], act=ops.ACT_RELU, alpha=al)
                eh, el = ops.split16(e.view(n * k, 400), scale=sa)
                pre = ops.linear_x3(eh, el, P[name + "_a1_hi"], P[name + "_a1_lo"], att.affine1.bias.detach(), alpha=al)
            else:
                e = ops.linear(feat, P["intent_w"], P["intent_b"], act=ops.ACT_RELU)          # [n, k*400]
                pre = ops.linear(e.view(n * k, 400), att.affine1.weight.detach(), att.affine1.bias.detach())
            out = torch.empty(n, 400, **f32)
            ops.intent_pool(pre, e, att.affine2.weight.detach().reshape(-1), out, n, k, 400)
            pooled.append(out)
        content = torch.empty(n, 900, **f32)
        ops.content_fuse(pooled[0], pooled[1], base.category_embedding.weight.detach(),
                         base.subCategory_embedding.weight.detach(), category, subCategory, content)
        return content

    def freshness_table(self):
        """T[bf*nb+bl] = W_f tanh(dense(E_f[bf] | E_l[bl])) + project.bias  -> [nb*nb, 400]
        (FreshnessEncoder.forward :60-83 followed by the freshness half of LIME.project :151-153)."""
        P = self.prepare()
        fe = self.m.freshness_encoder
        nb = fe.num_buckets
        dev = P["Wc"].device
        pairs = torch.empty(nb * nb, 2 * fe.freshness_embedding.weight.shape[1], dtype=torch.float32, device=dev)
        ops.bucket_pairs(fe.freshness_embedding.weight.detach(), fe.lifetime_embedding.weight.detach(), pairs)
        hid = ops.linear(pairs, fe.dense.weight.detach(), fe.dense.bias.detach(), act=ops.ACT_TANH)
        return ops.linear(hid, P["Wf"], P["proj_b"])


class ScoringEngine:
    """Stage B: folded user-encoder weights, cache rows, fused scoring launch."""

    def __init__(self, model):
        self.model = model
        self.cfg = model.config
        self.news = model.news_encoder.engine
        self._fold = None
        self._fp = None
        self._reset_topics()

    def _params(self):
        return [p for p in self.model.parameters()] + [b for b in self.model.buffers()]

    # -- topic registry: compact ids of the (category, subCategory) pairs seen so far + logit table ----
    def _reset_topics(self):
        self._topic_ids = {}          # (category, subCategory) key -> compact id
        self._topic_vec = []          # [52] topic representation per id (device)
        self._topic_tq = []           # [510] candidate-role affine image per id (device)
        self._topic_table = None      # [T, T, 12] exponentials of the head logits, rebuilt when the registry grows
        self._topic_table_n = 0
        self._topic_absmax = 0.0

    def _register_topics(self, category, subCategory, hist, cand):
        """Assign compact topic ids to the news of freshly built cache rows and stamp them into the
        rows (index building: torch plumbing; the logit table itself comes from lime_topic_pair_table)."""
        key = category.long() * 1000003 + subCategory.long()
        uniq, inverse = torch.unique(key, return_inverse=True)
        first = torch.full((uniq.numel(),), key.numel(), dtype=torch.long, device=key.device)
        first.scatter_reduce_(0, inverse, torch.arange(key.numel(), device=key.device), reduce="amin")
        lut = []
        for k, r in zip(uniq.tolist(), first.tolist()):
            if k not in self._topic_ids:
                self._topic_ids[k] = len(self._topic_ids)
                self._topic_vec.append(hist[r, HIST_T:HIST_T + TOPIC_LD].clone())
                self._topic_tq.append(cand[r, CAND_TQ:CAND_TQ + TOPIC * HEADS + HEADS].clone())
            lut.append(self._topic_ids[k])
        ids = torch.tensor(lut, dtype=torch.int32, device=key.device)[inverse]
        hist[:, HIST_TOPIC_ID].view(torch.int32).copy_(ids)
        cand[:, CAND_TOPIC_ID].view(torch.int32).copy_(ids)

    def topic_table(self):
        """(table [T,T,12] or None, T).  None when more than MAX_TOPICS topics are registered: the
        tensor-core scoring path is then unavailable and lime_score_impressions runs the exact kernel."""
        T = len(self._topic_ids)
        if T == 0 or T > MAX_TOPICS:
            return None, 0
        if self._topic_table is None or self._topic_table_n != T:
            lib = _lib.require_device()
            tv, tq = torch.stack(self._topic_vec).contiguous(), torch.stack(self._topic_tq).contiguous()
            tab = torch.empty(T, T, TOPIC_TAB_LD, dtype=torch.float32, device=tv.device)
            check(lib.lime_topic_pair_table(tv.data_ptr(), tv.stride(0), tq.data_ptr(), tq.stride(0), T,
                                            tab.data_ptr(), torch.cuda.current_stream().cuda_stream),
                  "lime_topic_pair_table")
            self._topic_table, self._topic_table_n = tab, T
            self._topic_absmax = float(tab.log2().abs().max())      # max |log2(e)-scaled logit|; one scalar per registry change (host read)
        return self._topic_table, T

    # -- fold the user-encoder weights (once per checkpoint) ---------------------------------------
    def fold(self):
        fp = _fingerprint(self._params())
        if self._fold is not None and fp == self._fp:
            return self._fold
        self._reset_topics()          # cached topic vectors belong to the previous weights
        ue = self.model.user_encoder
        ca = ue.candidate_aware_attn
        sage = ue.graph_sage.convs[0]
        dev = ue.K.weight.device
        f32 = dict(dtype=torch.float32, device=dev)
        WK, WQ, bQ = ue.K.weight.detach(), ue.Q.weight.detach(), ue.Q.bias.detach()
        Wl, bl, Wr = sage.lin_l.weight.detach(), sage.lin_l.bias.detach(), sage.lin_r.weight.detach()
        gamma, beta = ca.layernorm.weight.detach(), ca.layernorm.bias.detach()
        inv_s = 1.0 / math.sqrt(float(self.cfg.attention_dim))           # userEncoders.py:71,163
        F = {}
        # P = (W_K W_r)^T W_Q = W_r^T (W_K^T W_Q)
        X = ops.gemm_strided(WK.t(), WQ)
        Pm = ops.gemm_strided(Wr.t(), X)
        G = torch.zeros(CAND_NFOLD + 1, D, **f32)                       # [1208, 400], last row unused
        G[0:400].copy_(Pm)
        ops.scale_rows(G[0:400], gamma, inv_s)
        G[400:800].copy_(Wr.t())
        ops.scale_rows(G[400:800], gamma, 1.0)
        G[800:1200].copy_(Wl.t())
        ops.scale_rows(G[800:1200], gamma, 1.0)
        # LayerNorm subtracts the row mean of o, so only the mean-free part of each folded candidate
        # vector matters:  sum_d (o_d - mu) w_d = sum_d o_d (w_d - mean(w)).  Centring the three blocks
        # here (w -> (I - 11^T/D) w, linear in v) removes the cancellation D - mu * sum(w) from both
        # scoring kernels; the three "sum of w" scalars (columns 1200..1202) become exact zeros.
        centre = torch.eye(D, **f32) - 1.0 / D
        for blk in range(3):
            G[blk * 400:(blk + 1) * 400].copy_(ops.gemm_strided(centre, G[blk * 400:(blk + 1) * 400].clone()))
        ops.gemm_strided(beta.view(1, D), Pm, alpha=inv_s, out=G[1203:1204])   # B1 = beta . p / 20
        ops.gemm_strided(beta.view(1, D), Wr.t(), out=G[1204:1205])      # B2
        ops.gemm_strided(beta.view(1, D), Wl.t(), out=G[1205:1206])      # B3
        G[1206].copy_(bl)                                                # cb = b_l . c
        F["G"] = G
        # constants from Q.bias: p0 = W_r^T W_K^T b_Q
        x0 = ops.gemm_strided(bQ.view(1, D), WK)
        p0 = ops.gemm_strided(x0, Wr)                                    # [1, 400]
        cconst = torch.zeros(CAND_NFOLD + 1, **f32)
        cconst[0:400].copy_(p0.view(-1))
        ops.scale_rows(cconst[0:400].view(D, 1), gamma, inv_s)           # gamma * p0 / 20
        cconst[0:400].copy_(ops.gemm_strided(centre, cconst[0:400].clone().view(D, 1)).view(-1))
        ops.gemm_strided(beta.view(1, D), p0.view(D, 1), alpha=inv_s, out=cconst[1203:1204].view(1, 1))
        F["cconst"] = cconst
        # gate: z' = -log2(e) (a W_g v + b_g)
        Gg = ca.gate_proj.weight.detach().clone()
        ops.scale_rows(Gg, None, -LOG2E)
        gb = ca.gate_proj.bias.detach().clone().view(1, D)
        ops.scale_rows(gb, None, -LOG2E)
        F["Gg"], F["gate_bias"] = Gg, gb.view(-1)
        # bf16 pairs of the two per-news fold matrices (the tensor-core modes of Stage A run them as fp32x3 passes)
        for name in ("G", "Gg"):
            F[name + "_hi"], F[name + "_lo"] = ops.split16(F[name], scale=ops.X3_W_SCALE)
        # topic attention: S[head,h] = (W_k,head^T Q_head) . t_h + Q_head . b_k,head, all / sqrt(D),
        # with Q = W_q t_c + b_q   (layers.py:66-70)  ->  affine map of t_c into [50*10 + 10]
        Wq, bq = ca.query_proj.weight.detach(), ca.query_proj.bias.detach()
        Wk, bk = ca.key_proj.weight.detach(), ca.key_proj.bias.detach()
        hd = D // HEADS
        inv_sc = 1.0 / float(ca.scale)
        A = torch.zeros(TOPIC * HEADS + HEADS, TOPIC_LD, **f32)
        a0 = torch.zeros(TOPIC * HEADS + HEADS, **f32)
        Av = A[:TOPIC * HEADS].view(TOPIC, HEADS, TOPIC_LD)
        a0v = a0[:TOPIC * HEADS].view(TOPIC, HEADS)
        for h in range(HEADS):
            sl = slice(h * hd, (h + 1) * hd)
            ops.gemm_strided(Wk[sl].t(), Wq[sl], alpha=inv_sc, out=Av[:, h, :TOPIC])
            ops.gemm_strided(Wk[sl].t(), bq[sl].view(hd, 1), alpha=inv_sc, out=a0v[:, h:h + 1])
            r = TOPIC * HEADS + h
            ops.gemm_strided(bk[sl].view(1, hd), Wq[sl], alpha=inv_sc, out=A[r:r + 1, :TOPIC])
            ops.gemm_strided(bk[sl].view(1, hd), bq[sl].view(hd, 1), alpha=inv_sc, out=a0[r:r + 1].view(1, 1))
        F["Atq"], F["atq0"] = A, a0
        # user-node rows of the GraphSAGE mean: prefix sums of lin_l(user_node_embedding) (no bias)
        un = ops.linear(ue.user_node_embedding.detach(), Wl)
        ops.prefix_rows(un)
        F["un_prefix"] = un
        # bucket-pair tables
        T = self.news.freshness_table()                                  # [nb*nb, 400]
        nb2 = T.shape[0]
        htab = torch.empty(nb2, HTAB_LD, **f32)
        htab[:, :D].copy_(T)
        ops.linear(htab[:, :D], Gg, out=htab[:, D:])
        ctab = torch.zeros(nb2, CTAB_LD, **f32)
        ops.linear(htab[:, :D], G, bias=cconst, out=ctab[:, :CAND_NFOLD], n=CAND_NFOLD)
        F["hist_tab"], F["cand_tab"] = htab, ctab
        F["hist_tab_rep"] = htab.unsqueeze(0).repeat(TAB_REPLICAS, 1, 1).contiguous()      # plumbing copy
        F["htab_vg"] = interleave_vg(htab).unsqueeze(0).repeat(TAB_REPLICAS, 1, 1).contiguous()
        tabmax = torch.empty(2, nb2, **f32)
        ops.row_absmax(htab[:, D:], tabmax[0])
        F["ctab16"] = ops.split_f16_pairs(ctab, 3, absmax=tabmax[1])
        tm = tabmax.max(dim=1).values.tolist()          # two scalars per checkpoint (host read at fold time)
        F["tab_gw_absmax"] = tm[0]
        F["tc_tables_ok"] = int(tm[1] <= F16_SAFE)
        self._fold, self._fp = F, fp
        return F

    # -- per-news cache ----------------------------------------------------------------------------
    def build_rows(self, title_text, body_text, category, subCategory, chunk=2048):
        """Encode news and derive both cache roles.  int32 device tensors [n,32], [n,128], [n], [n]
        -> (hist_rows [n,852], cand_rows [n,1720])."""
        F = self.fold()
        lime = self.model.news_encoder
        n = title_text.shape[0]
        dev = title_text.device
        hist = torch.zeros(n, HIST_LD, dtype=torch.float32, device=dev)
        cand = torch.zeros(n, CAND_LD, dtype=torch.float32, device=dev)
        Wc = self.news.prepare()["Wc"]
        for lo in range(0, n, chunk):
            hi = min(n, lo + chunk)
            tt, bt = title_text[lo:hi].contiguous(), body_text[lo:hi].contiguous()
            ct, sb = category[lo:hi].contiguous(), subCategory[lo:hi].contiguous()
            content = self.news.encode_content(tt, bt, ct, sb)
            h, c = hist[lo:hi], cand[lo:hi]
            tc_mode = self.news.bf16 or self.news.x3        # tensor-core modes: the two folds as fp32x3 passes (2^-22 per product)
            al = 1.0 / (ops.X3_ACT_SCALE * ops.X3_W_SCALE)
            if tc_mode and self.news.x3_small:
                P = self.news.prepare()
                ch_, cl_ = ops.split16(content, scale=ops.X3_ACT_SCALE)
                ops.linear_x3(ch_, cl_, P["Wc_hi"], P["Wc_lo"], out=h[:, :D], alpha=al)   # vc
            else:
                ops.linear(content, Wc, out=h[:, :D])                               # vc
            if tc_mode:
                vh, vl = ops.split16(h[:, :D], scale=ops.X3_ACT_SCALE)
                ops.linear_x3(vh, vl, F["Gg_hi"], F["Gg_lo"], out=h[:, HIST_GW:HIST_GW + D], alpha=al)
            else:
                ops.linear(h[:, :D], F["Gg"], out=h[:, HIST_GW:HIST_GW + D])        # gw
            ops.topic_rep(lime.category_embedding.weight.detach(), lime.subCategory_embedding.weight.detach(),
                          lime.category_affine.weight.detach(), lime.category_affine.bias.detach(),
                          ct, sb, h[:, HIST_T:], TOPIC_LD)
            if tc_mode:
                ops.linear_x3(vh, vl, F["G_hi"], F["G_lo"], out=c[:, :CAND_NFOLD], n=CAND_NFOLD, alpha=al)
            else:
                ops.linear(h[:, :D], F["G"], out=c[:, :CAND_NFOLD], n=CAND_NFOLD)   # w1 w2 w3 + scalars
            ops.linear(h[:, HIST_T:HIST_T + TOPIC_LD], F["Atq"], F["atq0"],
                       out=c[:, CAND_TQ:CAND_TQ + TOPIC * HEADS + HEADS])           # tq, qb
        ops.row_absmax(hist[:, HIST_GW:HIST_GW + D], hist[:, HIST_GW_ABSMAX])
        self._register_topics(category, subCategory, hist, cand)
        return hist, cand

    def _score_long(self, hist_rows, cand_rows, dimp, ch, prefix_main, tail_start, prefix_tail, pair_index_base, out, cand16, meta, hist_vg):
        """Histories longer than the tensor-core kernel's 56 slots: lime_score_impressions_long on the chunked twin of ``dimp``."""
        lib = _lib.require_device()
        cache = self.cache_struct(hist_rows, cand_rows, cand16, meta, hist_vg)
        self._keepalive = (cand16, meta, hist_vg)
        if out is None:
            out = torch.empty(dimp.num_pairs, dtype=torch.float32, device=hist_rows.device)
        if tail_start is None:
            tail_start, prefix_tail = 1 << 62, prefix_main
        check(lib.lime_score_impressions_long(cache, dimp.struct(), ch.struct(), ch.chunks, dimp.num_pairs, dimp.num_impressions,
                                              int(pair_index_base), int(prefix_main), int(tail_start), int(prefix_tail), out.data_ptr(),
                                              ch.long_scratch.data_ptr(), ch.long_work.data_ptr(),
                                              torch.cuda.current_stream().cuda_stream), "lime_score_impressions_long")
        dimp.work_counter[:4].copy_(ch.long_scratch[:4])          # the caller reads the fallback count there
        return out

    def split_candidates(self, cand_rows):
        """cand16 [n + nb*nb, 2400] fp16: the folded candidate vectors as hi/lo pairs, followed by the nb*nb
        bucket-pair rows (ctab16) -- one operand array, so the scoring kernel addresses candidate rows and
        bucket-pair rows alike; stamps max |w| of every row into cand_rows[:, 1207] (the scoring kernel sends
        rows beyond the fp16 range to the exact kernel)."""
        F = self.fold()
        n, nb2 = cand_rows.shape[0], F["ctab16"].shape[0]
        c16 = torch.empty(n + TAB_REPLICAS * nb2, 2400, dtype=torch.float16, device=cand_rows.device)
        ops.split_f16_pairs(cand_rows, 3, absmax=cand_rows[:, CAND_ABSMAX], out=c16[:n])
        c16[n:].view(TAB_REPLICAS, nb2, 2400).copy_(F["ctab16"].unsqueeze(0).expand(TAB_REPLICAS, nb2, 2400))
        return c16

    @staticmethod
    def news_meta(hist_rows, cand_rows):
        """[n, 8] fp32, one 32-byte sector per news: topic id (int32 bits) | gw absmax | w absmax | B1 B2 B3 cb | 0 --
        the scalars phase 0 of the tensor-core kernel reads (column gather of existing cache values: plumbing).
        Call after split_candidates (which stamps the w absmax column)."""
        meta = torch.zeros(hist_rows.shape[0], 8, dtype=torch.float32, device=hist_rows.device)
        meta[:, 0:2].copy_(hist_rows[:, HIST_TOPIC_ID:HIST_GW_ABSMAX + 1])
        meta[:, 2].copy_(cand_rows[:, CAND_ABSMAX])
        meta[:, 3:7].copy_(cand_rows[:, CAND_SCAL + 3:CAND_SCAL + 7])
        return meta

    def cache_struct(self, hist_rows, cand_rows, cand16=None, meta=None, hist_vg=None):
        F = self.fold()
        cfg = self.cfg
        table, T = self.topic_table()
        return LimeNewsCache(
            hist_rows=hist_rows.data_ptr(), cand_rows=cand_rows.data_ptr(),
            hist_tab=F["hist_tab_rep"].data_ptr(), cand_tab=F["cand_tab"].data_ptr(), tab_replicas=TAB_REPLICAS,
            gate_bias=F["gate_bias"].data_ptr(), un_prefix=F["un_prefix"].data_ptr(),
            topic_table=table.data_ptr() if table is not None else None, num_topics=T,
            cand16=cand16.data_ptr() if cand16 is not None else None, ctab16=F["ctab16"].data_ptr(),
            news_meta=meta.data_ptr() if meta is not None else None,
            hist_vg=hist_vg.data_ptr() if hist_vg is not None else None, htab_vg=F["htab_vg"].data_ptr(),
            topic_logit_absmax=self._topic_absmax, tc_tables_ok=F["tc_tables_ok"],
            tab_gw_absmax=F["tab_gw_absmax"],
            news_num=hist_rows.shape[0], num_buckets=cfg.num_buckets,
            user_nodes=F["un_prefix"].shape[0], sigmoid_alpha=float(cfg.sigmoid_scaling_alpha),
            penalty_beta=float(cfg.penalty_scaling_beta),
            use_lifetime_weighting=int(bool(cfg.use_remaining_lifetime_weighting)),
            use_expired_penalty=int(bool(cfg.use_expired_penalty)))

    def lime_vectors(self, hist_rows, freshness, lifetime):
        """v = vc + T[bucket(freshness), bucket(lifetime)]  (LIME.forward output, [n,400])."""
        F = self.fold()
        nb = self.cfg.num_buckets
        idx = ops.bucketize(freshness, nb).long() * nb + ops.bucketize(lifetime, nb).long()
        # pure gather + add of two cached rows: plumbing for the module-level API, not on the scoring path
        return hist_rows[:, :D] + F["hist_tab"][:, :D].index_select(0, idx.reshape(-1))

    def score(self, hist_rows, cand_rows, dimp, prefix_main, tail_start=None, prefix_tail=None,
              pair_index_base=0, out=None, cand16=None, meta=None, hist_vg=None):
        """Launch the fused scoring kernel over a DeviceImpressions set -> fp32 scores [P].
        ``cand16`` / ``meta``: split_candidates(cand_rows) and news_meta(hist_rows, cand_rows) if the caller keeps
        them (NewsVectorCache does); derived here otherwise."""
        lib = _lib.require_device()
        if (cand16 is None or meta is None or hist_vg is None) and dimp.max_history <= TC_MAX_HISTORY:
            cand16 = self.split_candidates(cand_rows)
            meta = self.news_meta(hist_rows, cand_rows)
            hist_vg = interleave_vg(hist_rows)
        if getattr(dimp, "planned_buckets", None) is not None:
            dimp.replan(self.cfg.num_buckets)         # the unit list follows the model's bucketisation
        if dimp.max_history > TC_MAX_HISTORY and cand16 is not None and ops.score_mode() != ops.SCORE_EXACT:
            ch = dimp.chunked(self.cfg.num_buckets) if hasattr(dimp, "chunked") else None
            if ch is not None:
                return self._score_long(hist_rows, cand_rows, dimp, ch, prefix_main, tail_start, prefix_tail, pair_index_base, out,
                                        cand16, meta, hist_vg)
        cache = self.cache_struct(hist_rows, cand_rows, cand16, meta, hist_vg)
        self._keepalive = (cand16, meta, hist_vg)      # derived operands stay referenced until the next call (the launch is asynchronous)
        st = dimp.struct()
        if out is None:
            out = torch.empty(dimp.num_pairs, dtype=torch.float32, device=hist_rows.device)
        if tail_start is None:
            tail_start, prefix_tail = 1 << 62, prefix_main
        check(lib.lime_score_impressions(cache, st, int(pair_index_base), int(prefix_main), int(tail_start),
                                         int(prefix_tail), out.data_ptr(), dimp.work_counter.data_ptr(),
                                         torch.cuda.current_stream().cuda_stream), "lime_score_impressions")
        return out


def choose_tile_c(max_history):
    """Candidates per work unit for this history length (lime_score_tile_c: 42 on the tensor-core
    path, H <= 64; the largest shared-memory-feasible multiple of 8 up to 48 on the exact path)."""
    lib = _lib.load()
    tc = int(lib.lime_score_tile_c(int(max_history)))
    if tc <= 0:
        raise _lib.LimeError("max_history=%d does not fit the scoring kernel's shared memory" % max_history)
    return tc


def _host_bucket_pairs(fresh, life, nb):
    """Approximate (freshness, lifetime) bucket pair per candidate on the host -- used ONLY to size work units (how many
    distinct pairs a run of candidates holds); the scoring kernel derives the exact buckets itself and sends a unit that
    still does not fit to the exact kernel, so a knife-edge disagreement costs speed, never correctness."""
    def b(x):
        x = np.maximum(np.asarray(x, np.float32), np.float32(1.0))
        v = np.log(x).astype(np.float32) * np.float32(1.0 / math.log(86400.0)) * np.float32(nb / 7.0)
        return np.clip(v.astype(np.int64), 0, nb - 1)
    return b(fresh) * nb + b(life)


def build_units(cand_off, tile_c, cand_bp=None, triples=None, max_pairs=20):
    """Work units of the scoring kernel: every impression's candidate list is cut into runs of consecutive candidates.
    Without ``cand_bp``: runs of at most ``tile_c``.  With ``cand_bp`` (bucket-pair id per candidate) and ``triples``
    (operand-row triples of the tensor-core kernel, 40): greedy runs with candidates + distinct bucket pairs <= triples
    (the pairs ride along as extra operand rows) and at most ``max_pairs`` distinct pairs (the kernel's kMaxBp), at most
    ``tile_c`` candidates.
    Returns (unit_imp, unit_pair0, unit_count) as int64."""
    cand_off = np.asarray(cand_off, np.int64)
    counts = np.diff(cand_off)
    if cand_bp is None:
        nun = (counts + tile_c - 1) // tile_c
        unit_imp = np.repeat(np.arange(counts.shape[0], dtype=np.int64), nun)
        first = np.cumsum(nun) - nun
        kk = np.arange(unit_imp.shape[0], dtype=np.int64) - first[unit_imp]
        unit_pair0 = cand_off[:-1][unit_imp] + kk * tile_c
        unit_count = np.minimum(tile_c, counts[unit_imp] - kk * tile_c)
        return unit_imp, unit_pair0, unit_count
    cand_bp = np.asarray(cand_bp, np.int64)
    ui, up, uc = [], [], []
    # impressions whose candidates + (at most that many) pairs fit one unit need no scan
    safe = (2 * counts <= triples) & (counts <= max_pairs)
    for i in range(counts.shape[0]):
        n, o = int(counts[i]), int(cand_off[i])
        if n == 0:
            continue
        if safe[i]:
            ui.append(i); up.append(o); uc.append(n)
            continue
        b = cand_bp[o:o + n].tolist()
        j = 0
        while j < n:
            seen, c = set(), 0
            while j + c < n and c < tile_c:
                x = b[j + c]
                if c + 1 + len(seen) + (x not in seen) > triples or len(seen) + (x not in seen) > max_pairs:
                    break
                seen.add(x)
                c += 1
            c = max(c, 1)
            ui.append(i); up.append(o + j); uc.append(c)
            j += c
    return np.asarray(ui, np.int64), np.asarray(up, np.int64), np.asarray(uc, np.int64)


def plan_pool(bucket_pair, topic, limit):
    """Work-unit plan of a news pool scored against every user (torch, CPU or device).  bucket_pair [C] (the approximate
    (freshness, lifetime) bucket pair of _host_bucket_pairs) and topic [C] (compact topic id) -> (order, unit_pair0,
    unit_count), int64:
      order       a permutation of the pool: stable sort by (bucket pair, topic);
      unit_pair0  first plan position of every unit, unit_count its size: units never straddle a bucket-pair group and
                  hold at most ``limit`` candidates.
    A unit then carries one distinct bucket pair beside its <= limit candidates (the tensor-core kernel's 40 operand-row
    triples fit 39), and candidates of one topic have one candidate-aware attention vector (DESIGN.md section 3c), so the
    kernel's expansion around the unit's centre is exact and the unit stays off the exact-kernel fallback."""
    bp, tp = bucket_pair.long(), topic.long()
    C = bp.numel()
    if C == 0:
        e = torch.zeros(0, dtype=torch.long, device=bp.device)
        return e, e, e
    order = torch.sort((bp << 32) | tp, stable=True).indices
    sbp = bp[order]
    pos = torch.arange(C, device=bp.device)
    start = torch.ones(C, dtype=torch.bool, device=bp.device)
    start[1:] = sbp[1:] != sbp[:-1]
    first = torch.cummax(torch.where(start, pos, torch.zeros_like(pos)), 0).values     # first position of the group
    unit_pair0 = torch.nonzero((pos - first) % int(limit) == 0).squeeze(1)
    unit_count = torch.diff(unit_pair0, append=torch.tensor([C], device=bp.device))
    return order, unit_pair0, unit_count


class PoolPlan:
    """A news pool laid out for lime_score_impressions (recommend.plan builds it).  Device tensors, all in plan order:
    news / fresh / life [C] (cache row, seconds), remaining [C] or None (the remaining lifetime of lifetime_type 'fixed' /
    'topic_wise'), index [C] int32 (the caller's index of the position), exclude [C] uint8 or None, bucket_pair / topic
    [C] (the sort keys), and caller_news [C] int64 (the cache row of every caller index)."""

    def __init__(self, news, fresh, life, remaining, index, exclude, bucket_pair, topic, caller_news):
        self.news, self.fresh, self.life, self.remaining = news, fresh, life, remaining
        self.index, self.exclude, self.bucket_pair, self.topic = index, exclude, bucket_pair, topic
        self.caller_news = caller_news
        self.device = news.device
        self.templates = {}          # limit -> (unit_pair0, unit_count) int32 of one user
        self._positions = None

    @property
    def size(self):
        return int(self.news.numel())

    def positions(self, news_num):
        """[news_num] int32 device table: the plan position of every cache row, -1 = not in the pool (built once)."""
        if self._positions is None or self._positions.numel() != news_num:
            t = torch.full((news_num,), -1, dtype=torch.int32, device=self.device)
            t[self.news.long()] = torch.arange(self.size, dtype=torch.int32, device=self.device)
            self._positions = t
        return self._positions

    def units(self, limit):
        """The unit template of one user for at most ``limit`` candidates per unit (the plan order is plan_pool's)."""
        if limit not in self.templates:
            _, p0, cnt = plan_pool(self.bucket_pair, self.topic, limit)
            self.templates[limit] = (p0.to(torch.int32), cnt.to(torch.int32))
        return self.templates[limit]


class DeviceImpressions:
    """Impression set resident in HBM + the work-unit list of the scoring kernel."""

    @classmethod
    def from_pool(cls, plan, hist_news, hist_mask, hist_fresh, hist_life):
        """Every one of Ub users (histories [Ub, H], device tensors) against the whole pool of ``plan`` (a PoolPlan): impression
        u = user u, its candidates the pool in plan order (pair u * C + c).  Device tensors only, no host copies: the
        candidate arrays are expanded copies of the plan's, the unit list is the plan's template shifted by u * C.
        H <= 56 runs the tensor-core kernel; longer histories (up to 224) run the exact kernel, because the chunked
        tensor-core path (DeviceImpressions.chunked) is built from host arrays -- correct, but several times slower."""
        self = cls.__new__(cls)
        dev = hist_mask.device
        Ub, H = hist_mask.shape
        C = plan.size
        if Ub * C >= 2 ** 31:
            raise _lib.LimeError("from_pool: %d users x %d news exceed the int32 pair index" % (Ub, C))
        i32 = dict(dtype=torch.int32, device=dev)
        self.tile_c = choose_tile_c(H)
        p0, cnt = plan.units(min(self.tile_c, TC_TRIPLES - 2))     # room for one bucket-pair knife-edge per unit
        nu = p0.numel()
        self.max_history, self.num_pairs, self.num_impressions, self.num_units = H, Ub * C, Ub, Ub * nu
        self.device = dev
        self.planned_buckets = None
        u = torch.arange(Ub, **i32).view(Ub, 1)
        pairs = lambda t: t.view(1, C).expand(Ub, C).reshape(-1)
        self.dev = dict(
            hist_news=hist_news.to(torch.int32).contiguous(), hist_mask=hist_mask.to(torch.uint8).contiguous(),
            hist_fresh=hist_fresh.float().contiguous(), hist_life=hist_life.float().contiguous(),
            cand_news=pairs(plan.news), cand_fresh=pairs(plan.fresh), cand_life=pairs(plan.life),
            unit_imp=u.expand(Ub, nu).reshape(-1), unit_pair0=(p0.view(1, nu) + u * C).reshape(-1),
            unit_count=cnt.view(1, nu).expand(Ub, nu).reshape(-1))
        if plan.remaining is not None:
            self.dev["cand_remaining"] = pairs(plan.remaining)
        self.work_counter = torch.zeros(int(_lib.load().lime_score_scratch_ints(self.num_units)), **i32)
        return self

    @classmethod
    def from_pairs(cls, hist_mask, hist_fresh, hist_life, cand_fresh, cand_life, cand_remaining, n_cand):
        """Per-pair layout of Model.forward (one impression per sample, ``n_cand`` candidates each):
        the freshly encoded batch is its own news cache with history rows first
        (row b*H+h) and candidate rows after them (row B*H + b*n_cand + j).  Device tensors only."""
        self = cls.__new__(cls)
        dev = hist_mask.device
        B, H = hist_mask.shape
        i32 = dict(dtype=torch.int32, device=dev)
        self.tile_c = choose_tile_c(H)
        if n_cand > self.tile_c:
            raise _lib.LimeError("at most %d candidates per sample in Model.forward" % self.tile_c)
        self.max_history, self.num_pairs, self.num_impressions, self.num_units = H, B * n_cand, B, B
        self.device = dev
        self.dev = dict(
            hist_news=torch.arange(B * H, **i32).view(B, H),
            hist_mask=hist_mask.to(torch.uint8).contiguous(),
            hist_fresh=hist_fresh.float().contiguous(), hist_life=hist_life.float().contiguous(),
            cand_news=torch.arange(B * H, B * H + B * n_cand, **i32),
            cand_fresh=cand_fresh.float().reshape(-1).contiguous(),
            cand_life=cand_life.float().reshape(-1).contiguous(),
            unit_imp=torch.arange(B, **i32), unit_pair0=torch.arange(0, B * n_cand, n_cand, **i32),
            unit_count=torch.full((B,), n_cand, **i32))
        if cand_remaining is not None:
            self.dev["cand_remaining"] = cand_remaining.float().reshape(-1).contiguous()
        self.work_counter = torch.zeros(int(_lib.load().lime_score_scratch_ints(self.num_units)), dtype=torch.int32, device=dev)
        return self

    def __init__(self, imp, device, tile_c=None, cand_remaining=None, num_buckets=10):
        H = imp.hist_news.shape[1]
        self.tile_c = int(tile_c or choose_tile_c(H))
        self.max_history = H
        self.num_pairs = int(imp.cand_news.shape[0])
        self.num_impressions = int(imp.hist_news.shape[0])
        self._fixed_tile = tile_c is not None
        self.planned_buckets = None
        if H <= TC_MAX_HISTORY and tile_c is None and num_buckets is not None:
            # tensor-core path: a unit's candidates and its distinct bucket pairs share the 40 operand-row triples
            bp = _host_bucket_pairs(imp.cand_fresh, imp.cand_life, int(num_buckets))
            unit_imp, unit_pair0, unit_count = build_units(imp.cand_off, self.tile_c, bp, TC_TRIPLES)
            self.planned_buckets = int(num_buckets)
        else:
            unit_imp, unit_pair0, unit_count = build_units(imp.cand_off, self.tile_c)
        self.num_units = int(unit_imp.shape[0])
        self.host = dict(
            hist_news=np.ascontiguousarray(imp.hist_news, np.int32),
            hist_mask=np.ascontiguousarray(imp.hist_mask).astype(np.uint8),
            hist_fresh=np.ascontiguousarray(imp.hist_fresh, np.float32),
            hist_life=np.ascontiguousarray(imp.hist_life, np.float32),
            cand_news=np.ascontiguousarray(imp.cand_news, np.int32),
            cand_fresh=np.ascontiguousarray(imp.cand_fresh, np.float32),
            cand_life=np.ascontiguousarray(imp.cand_life, np.float32),
            unit_imp=unit_imp.astype(np.int32), unit_pair0=unit_pair0.astype(np.int32),
            unit_count=unit_count.astype(np.int32),
            cand_off=np.ascontiguousarray(imp.cand_off, np.int64),
            labels=np.ascontiguousarray(imp.labels, np.uint8),
        )
        if cand_remaining is not None:      # lifetime_type 'fixed' / 'topic_wise' (util.py:98-102)
            self.host["cand_remaining"] = np.ascontiguousarray(cand_remaining, np.float32)
        self.pinned = {k: torch.from_numpy(v).pin_memory() for k, v in self.host.items()}
        self.dev = {}
        self.device = device
        self.work_counter = torch.zeros(int(_lib.load().lime_score_scratch_ints(self.num_units)), dtype=torch.int32,
                                        device=device)
        self.upload()

    def replan(self, num_buckets):
        """Rebuild the unit list for a model with ``num_buckets`` lifetime buckets (the planner packs candidates + distinct
        bucket pairs into a unit, so the bucketisation must be the model's: a list planned for another bucket count is
        still scored correctly, but its over-full units all take the exact-kernel fallback)."""
        if self._fixed_tile or self.max_history > TC_MAX_HISTORY or self.planned_buckets == int(num_buckets) or "cand_off" not in self.host:
            return
        bp = _host_bucket_pairs(self.host["cand_fresh"], self.host["cand_life"], int(num_buckets))
        unit_imp, unit_pair0, unit_count = build_units(self.host["cand_off"], self.tile_c, bp, TC_TRIPLES)
        self.planned_buckets = int(num_buckets)
        self.num_units = int(unit_imp.shape[0])
        for k, v in (("unit_imp", unit_imp), ("unit_pair0", unit_pair0), ("unit_count", unit_count)):
            self.host[k] = v.astype(np.int32)
            self.pinned[k] = torch.from_numpy(self.host[k]).pin_memory()
            self.dev[k] = self.pinned[k].to(self.device, non_blocking=True)
        self.work_counter = torch.zeros(int(_lib.load().lime_score_scratch_ints(self.num_units)), dtype=torch.int32, device=self.device)

    def chunked(self, num_buckets):
        """The twin of a long-history set (H > 56) for lime_score_impressions_long: every impression cut into K pieces of
        H / K <= 56 slots (pseudo-impression k * I + i), candidates replicated chunk-major; None if H does not divide."""
        H = self.max_history
        if getattr(self, "_chunked", None) is not None and self._chunked.planned_buckets == int(num_buckets):
            return self._chunked
        if "cand_off" not in getattr(self, "host", {}) or "cand_remaining" in self.host:
            return None
        K = next((k for k in range((H + TC_MAX_HISTORY - 1) // TC_MAX_HISTORY, H + 1) if H % k == 0 and H // k <= TC_MAX_HISTORY), None)
        if K is None or H // K < 8:
            return None
        from .synth import Impressions
        h, I_, Hc, P = self.host, self.num_impressions, H // K, self.num_pairs
        cut = lambda a: np.ascontiguousarray(np.transpose(a.reshape(I_, K, Hc), (1, 0, 2)).reshape(K * I_, Hc))
        off = np.concatenate([h["cand_off"][:-1] + k * P for k in range(K)] + [np.asarray([K * P], np.int64)])
        imp = Impressions(cut(h["hist_news"]), cut(h["hist_mask"]), cut(h["hist_fresh"]), cut(h["hist_life"]), off,
                          np.tile(h["cand_news"], K), np.tile(h["cand_fresh"], K), np.tile(h["cand_life"], K),
                          np.tile(h["labels"], K), np.zeros(K * I_, np.int64))
        ch = DeviceImpressions(imp, self.device, num_buckets=int(num_buckets))
        lib = _lib.load()
        ch.chunks = K
        ch.long_scratch = torch.zeros(int(lib.lime_score_long_scratch_ints(ch.num_units, self.num_units)), dtype=torch.int32, device=self.device)
        ch.long_work = torch.empty(int(lib.lime_score_long_work_floats(P, H, K)), dtype=torch.float32, device=self.device)
        self._chunked = ch
        return ch

    def h2d_bytes(self):
        return int(sum(v.numel() * v.element_size() for v in self.pinned.values()))

    def upload(self):
        """Host (pinned) -> HBM copy of every input array, on the current stream."""
        for k, v in self.pinned.items():
            if k not in self.dev:
                self.dev[k] = torch.empty(v.shape, dtype=v.dtype, device=self.device)
            self.dev[k].copy_(v, non_blocking=True)

    def struct(self):
        d = self.dev
        return LimeImpressions(
            hist_news=d["hist_news"].data_ptr(), hist_mask=d["hist_mask"].data_ptr(),
            hist_fresh=d["hist_fresh"].data_ptr(), hist_life=d["hist_life"].data_ptr(),
            cand_news=d["cand_news"].data_ptr(), cand_fresh=d["cand_fresh"].data_ptr(),
            cand_life=d["cand_life"].data_ptr(),
            cand_remaining=d["cand_remaining"].data_ptr() if "cand_remaining" in d else None,
            unit_imp=d["unit_imp"].data_ptr(),
            unit_pair0=d["unit_pair0"].data_ptr(), unit_count=d["unit_count"].data_ptr(),
            num_units=self.num_units, max_history=self.max_history, tile_c=self.tile_c)
