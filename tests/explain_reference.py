"""fp64-capable reference of recommend.explain for the tests: oracle.score_from_vectors with the score split into one term
per history slot.  Test infrastructure like oracle/lime_oracle.py, built from its functions (crown_user restated term by
term); kept beside the tests that use it so the pinned oracle module stays as it is."""
import math

import numpy as np
import torch

from oracle.lime_oracle import NEWS, USER, _lin, candidate_aware_attention, lifetime_weight, topic_representation


def explain_from_vectors(sd, cfg, hist_vec, hist_cat, hist_sub, hist_mask, cand_vec, cand_cat, cand_sub, remaining, prefix,
                         dtype=torch.float32, group=64):
    """score_from_vectors (same arguments) with the score split into one term per history slot: crown_user restated term by
    term.  With x_h the history rows after candidate_aware_attention, g_h = lin_l(m) + lin_r(x_h) and m the mean of the
    first P rows of [x ; user_node_embedding] (userEncoders.py:121,151-157), alpha = softmax_h(Q(c) . K(g_h) / sqrt(A))
    (:161-164) and w = lifetime_weight(remaining) (util.py:39-48):
        score = w ((alpha @ g) . c) = bias + sum_h contrib[h]
        contrib[h] = w (alpha_h x_h . W_r^T c + [h < min(P, H)] x_h . W_l^T c / P)
        bias = w (b_l . c + (1/P) sum_{j < P - H} user_node_j . W_l^T c)
    -> dict of alpha / topic_attention (the candidate-aware weights, layers.py:81; NaN when the model has no
    candidate-aware attention) / contrib [N, H], bias / weight / score [N] in ``dtype`` (score from alpha @ g, as
    crown_user computes it)."""
    H, D = hist_vec.shape
    N = cand_vec.shape[0]
    hv, cv = hist_vec.to(dtype), cand_vec.to(dtype)
    hc, hs, hm = (torch.as_tensor(np.asarray(x)) for x in (hist_cat, hist_sub, hist_mask))
    cc, cs = torch.as_tensor(np.asarray(cand_cat)), torch.as_tensor(np.asarray(cand_sub))
    pre = np.broadcast_to(np.asarray(prefix, np.int64), (N,))
    S = USER + "graph_sage.convs.0."
    Wl, bl, Wr = (sd[S + n].to(dtype) for n in ("lin_l.weight", "lin_l.bias", "lin_r.weight"))
    un = sd[USER + "user_node_embedding"].to(dtype)
    out = {n: torch.empty(N, H, dtype=dtype) for n in ("alpha", "topic_attention", "contrib")}
    out.update({n: torch.empty(N, dtype=dtype) for n in ("bias", "score")})
    for p in np.unique(pre).tolist():
        if p > H + un.shape[0]:
            raise IndexError("runtime batch %d exceeds max_history_num + config.batch_size = %d" % (p, H + un.shape[0]))
        sel = np.nonzero(pre == p)[0]
        for lo in range(0, sel.shape[0], group):
            idx = torch.as_tensor(sel[lo:lo + group])
            g = idx.numel()
            c = cv[idx]                                                               # [g, D]
            x = hv.unsqueeze(0).expand(g, H, D)
            ta = torch.full((g, H), float("nan"), dtype=dtype)
            if cfg.use_candidate_ware_clicked_news_attention:                         # :103-117
                x, ta = candidate_aware_attention(
                    sd, x, topic_representation(sd, NEWS, hc.view(1, H).expand(g, H), hs.view(1, H).expand(g, H), dtype),
                    topic_representation(sd, NEWS, cc[idx].view(g, 1), cs[idx].view(g, 1), dtype),
                    hm.view(1, H).expand(g, H).bool(), dtype)
            rows = torch.cat([x, un.unsqueeze(0).expand(g, -1, -1)], dim=1)          # :121
            m = rows[:, :p].mean(dim=1)                                               # GraphSAGE mean over the prefix
            xr = x @ Wr.t()
            gh = (m @ Wl.t() + bl).unsqueeze(1) + xr                                  # :151-157
            K = gh @ sd[USER + "K.weight"].to(dtype).t()                              # :161
            Q = _lin(c, sd, USER + "Q", dtype)                                        # :162
            alpha = torch.softmax((K @ Q.unsqueeze(-1)).squeeze(-1) / math.sqrt(float(cfg.attention_dim)), dim=-1)  # :163-164
            y = (xr @ c.unsqueeze(-1)).squeeze(-1)                                    # x_h . W_r^T c
            z = ((x @ Wl.t()) @ c.unsqueeze(-1)).squeeze(-1)                          # x_h . W_l^T c
            z = torch.where(torch.arange(H) < min(p, H), z, torch.zeros_like(z))
            unc = ((un[:max(p - H, 0)] @ Wl.t()).sum(dim=0).unsqueeze(0) * c).sum(dim=-1)   # user-node rows of the mean
            out["alpha"][idx], out["topic_attention"][idx] = alpha, ta
            out["contrib"][idx] = alpha * y + z / p
            out["bias"][idx] = (c @ bl) + unc / p
            out["score"][idx] = ((alpha.unsqueeze(-1) * gh).sum(dim=1) * c).sum(dim=-1)   # :168-169, util.py:32
    w = lifetime_weight(torch.as_tensor(np.asarray(remaining, np.float32)).to(dtype), cfg)
    out["weight"] = w
    out["contrib"] = out["contrib"] * w.unsqueeze(-1)
    out["bias"], out["score"] = out["bias"] * w, out["score"] * w
    return out


