"""Top-k news of a candidate pool for every user: the question a deployed recommender answers.

    plan = recommend.plan(model, cache, pool_news, pool_fresh, pool_life, exclude=None)      # once per pool state
    res = recommend.top_k(model, cache, plan, hist_news, hist_mask, hist_fresh, hist_life, k)
    res.index [U, k] int64 caller pool index (-1 pad), res.news [U, k] int64 cache row (-1 pad), res.score [U, k] fp32
    (-inf pad), res.count [U] int64, res.fallback_units (int: units the exact kernel re-scored; reading it synchronises)

Every user is scored against every pool news by lime_score_impressions (the pool is one impression per user, its work
units planned once per pool by engine.plan_pool), and lime_pool_topk keeps the k best per user, so only [U, k] leaves
the device.  Order: descending score, equal scores by ascending caller index -- the order lime_rank_metrics gives the
pool in the caller's order.  News the user clicked (masked-in history slots) are never returned with exclude_clicked,
nor are positions the plan's ``exclude`` marks, nor NaN scores.

Offline evaluation of the same lists: hold out each user's later clicks and rank them in the whole pool.

    ev = recommend.evaluate(model, cache, plan, hist_news, hist_mask, hist_fresh, hist_life, target_news, target_mask,
                            cutoffs=(10, 50, 100), exclude_clicked=True)
    ev.rank [U, T] int32 (1-based, 0 = unranked), ev.ranked [U] int32, ev.eligible [U] int64,
    ev.metrics [U, 4 + 2 len(cutoffs)] fp64 with names ev.columns, ev.means() -> dict, ev.fallback_units

A target's rank counts every position top_k could return to the user (other targets included), in top_k's order, so
rank r <= k means top_k(k) returns that news at position r.  lime_pool_rank_metrics ranks them on the device.

GraphSAGE semantics: every (user, news) pair is scored as it would be in a FULL mini-batch of config.batch_size of the
reference's eval loop (SURVEY.md section 8a row 10: the user-node prefix length follows the runtime batch size), so a
score depends on neither the pool's size or order nor on how users are batched.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib, ops
from .engine import HIST_TOPIC_ID, TC_TRIPLES, DeviceImpressions, PoolPlan, _host_bucket_pairs, plan_pool
from .util import remaining_lifetime

PAIR_BUDGET = 1 << 24        # (user, news) pairs per scoring launch: 64 MB of scores, far from the int32 pair index


def _host(a, dtype):
    return np.ascontiguousarray(a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a), dtype)


def _topic_categories(model):
    """Category id of every compact topic id of the model's registry (ScoringEngine._register_topics keys)."""
    ids = model.scoring._topic_ids
    cats = np.zeros(len(ids), np.int64)
    for key, tid in ids.items():
        cats[tid] = key // 1000003
    return cats


def validate_pool(news_num, pool_news, pool_fresh, pool_life, exclude=None):
    """Host-side checks of a pool: non-empty, equal lengths, ids in [1, news_num) and each at most once (a news is
    returned once), finite times.  -> the arrays as numpy (int32, fp32, fp32, uint8 or None)."""
    news = _host(pool_news, np.int64)
    fresh, life = _host(pool_fresh, np.float32), _host(pool_life, np.float32)
    if news.ndim != 1 or news.size == 0:
        raise ValueError("pool_news must be a non-empty 1-D array")
    if fresh.shape != news.shape or life.shape != news.shape:
        raise ValueError("pool_news, pool_fresh and pool_life must have the same length")
    if exclude is not None:
        exclude = _host(exclude, np.uint8)
        if exclude.shape != news.shape:
            raise ValueError("exclude must have one entry per pool news")
    if news.min() < 1 or news.max() >= news_num:
        raise ValueError("pool news ids must lie in [1, %d)" % news_num)
    if np.unique(news).size != news.size:
        raise ValueError("a pool lists every news at most once")
    if not (np.isfinite(fresh).all() and np.isfinite(life).all()):
        raise ValueError("pool_fresh / pool_life must be finite")
    if news.size >= 2 ** 31:
        raise ValueError("pool larger than 2^31 - 1 news")
    return news.astype(np.int32), fresh, life, exclude


def plan(model, cache, pool_news, pool_fresh, pool_life, exclude=None):
    """Lay a pool out for scoring (once per pool state): pool_news [C] cache rows, pool_fresh / pool_life [C] seconds
    (freshness at request time, lifetime), exclude [C] nonzero = never returned.  The pool is sorted by (approximate
    bucket pair, topic) -- ties by news id, so the plan does not depend on the caller's order -- and cut into units
    (engine.plan_pool).  -> engine.PoolPlan on the cache's device."""
    cfg = model.config
    news, fresh, life, exclude = validate_pool(cache.news_num, pool_news, pool_fresh, pool_life, exclude)
    dev = cache.hist_rows.device
    news_d = torch.from_numpy(news).to(dev)
    topic = cache.hist_rows[:, HIST_TOPIC_ID].view(torch.int32)[news_d.long()]
    remaining = remaining_lifetime(cfg, fresh, lambda: _topic_categories(model)[topic.cpu().numpy()])
    bp = torch.from_numpy(_host_bucket_pairs(fresh, life, int(cfg.num_buckets))).to(dev)
    by_news = torch.argsort(news_d, stable=True)
    limit = TC_TRIPLES - 2
    order, p0, cnt = plan_pool(bp[by_news], topic[by_news], limit)
    order = by_news[order]
    t = lambda a: torch.from_numpy(a).to(dev)[order].contiguous()
    p = PoolPlan(news=news_d[order].contiguous(), fresh=t(fresh), life=t(life),
                 remaining=t(remaining) if remaining is not None else None,
                 index=order.to(torch.int32).contiguous(), exclude=t(exclude) if exclude is not None else None,
                 bucket_pair=bp[order].contiguous(), topic=topic[order].contiguous(), caller_news=news_d.long())
    p.templates[limit] = (p0.to(torch.int32), cnt.to(torch.int32))
    return p


class TopK:
    """Result of top_k (device tensors; see the module docstring)."""

    def __init__(self, index, news, score, count, fallback):
        self.index, self.news, self.score, self.count = index, news, score, count
        self._fallback = fallback

    @property
    def fallback_units(self):
        return int(self._fallback)


def _histories(plan, hist_news, hist_mask, hist_fresh, hist_life):
    dev = plan.device
    dt = lambda a, dtype: (a if torch.is_tensor(a) else torch.from_numpy(np.asarray(a))).to(device=dev, dtype=dtype).contiguous()
    hn, hm = dt(hist_news, torch.int32), dt(hist_mask, torch.uint8)
    hf, hl = dt(hist_fresh, torch.float32), dt(hist_life, torch.float32)
    if hn.dim() != 2 or hm.shape != hn.shape or hf.shape != hn.shape or hl.shape != hn.shape:
        raise ValueError("hist_news / hist_mask / hist_fresh / hist_life must share one [users, max_history] shape")
    return hn, hm, hf, hl


def _scored_batches(model, cache, plan, hist, fallback):
    """Score every user of ``hist`` (device histories) against the whole pool, PAIR_BUDGET // C users per launch.
    Yields (u0, u1, scores [u1 - u0, C] in plan order); the buffer is reused by the next batch.  Units the exact kernel
    re-scored are added to the device counter ``fallback``."""
    hn, hm, hf, hl = hist
    U, C = hn.shape[0], plan.size
    ub = max(1, min(U, PAIR_BUDGET // C))
    scores = torch.empty(ub * C, dtype=torch.float32, device=plan.device)
    for u0 in range(0, U, ub):
        u1 = min(U, u0 + ub)
        dimp = DeviceImpressions.from_pool(plan, hn[u0:u1], hm[u0:u1], hf[u0:u1], hl[u0:u1])
        s = model.scoring.score(cache.hist_rows, cache.cand_rows, dimp, prefix_main=int(model.config.batch_size),
                                out=scores[:(u1 - u0) * C], cand16=cache.cand16, meta=cache.meta, hist_vg=cache.hist_vg)
        fallback += dimp.work_counter[1]
        yield u0, u1, s.view(u1 - u0, C)


def top_k(model, cache, plan, hist_news, hist_mask, hist_fresh, hist_life, k, exclude_clicked=True):
    """The k best news of ``plan``'s pool for each of U users: histories [U, H] (cache rows, mask, seconds; H <= 224,
    H > 56 runs the exact scoring kernel, several times slower), 1 <= k <= 1024.  Asynchronous: nothing is read back
    until the caller reads the result.  Users are scored in batches of PAIR_BUDGET / C; see the module docstring for
    what a score means."""
    if not 1 <= int(k) <= ops.TOPK_MAX:
        raise ValueError("k must lie in [1, %d]" % ops.TOPK_MAX)
    dev = plan.device
    hist = _histories(plan, hist_news, hist_mask, hist_fresh, hist_life)
    hn, hm = hist[0], hist[1]
    U, k = hn.shape[0], int(k)
    res = TopK(torch.full((U, k), -1, dtype=torch.int64, device=dev), torch.full((U, k), -1, dtype=torch.int64, device=dev),
               torch.full((U, k), float("-inf"), dtype=torch.float32, device=dev), torch.zeros(U, dtype=torch.int64, device=dev),
               torch.zeros((), dtype=torch.int64, device=dev))
    with torch.no_grad():
        for u0, u1, s in _scored_batches(model, cache, plan, hist, res._fallback):
            idx, val, cnt = ops.pool_topk(s, k, plan.index, plan.news, plan.exclude,
                                          hn[u0:u1] if exclude_clicked else None, hm[u0:u1] if exclude_clicked else None)
            idx = idx.long()
            res.index[u0:u1] = idx
            res.news[u0:u1] = torch.where(idx >= 0, plan.caller_news[idx.clamp_min(0)], -1)
            res.score[u0:u1] = val
            res.count[u0:u1] = cnt
    return res


class Evaluation:
    """Result of evaluate (device tensors; see the module docstring)."""

    def __init__(self, rank, ranked, eligible, metrics, columns, fallback):
        self.rank, self.ranked, self.eligible, self.metrics, self.columns = rank, ranked, eligible, metrics, columns
        self._fallback = fallback

    @property
    def fallback_units(self):
        return int(self._fallback)

    def means(self):
        """Mean of every metric column over the users with at least one ranked target (reads the device), and their
        number under "users".  An AUC of NaN (every eligible position a target) makes the mean AUC NaN."""
        m = self.metrics.cpu().numpy()[self.ranked.cpu().numpy() > 0]
        out = {c: float(m[:, i].mean()) if len(m) else float("nan") for i, c in enumerate(self.columns)}
        out["users"] = int(len(m))
        return out


def evaluate(model, cache, plan, hist_news, hist_mask, hist_fresh, hist_life, target_news, target_mask,
             cutoffs=(10, 50, 100), exclude_clicked=True):
    """Rank each user's held-out clicks in ``plan``'s whole pool, as top_k would order it: histories as in top_k,
    target_news [U, T] cache rows in [0, news_num) with target_mask [U, T] (T <= 256), cutoffs up to 8 ints >= 1 (the K
    of Recall@K and nDCG@K).  Masked slots, news not in the pool, excluded or clicked news, NaN scores and later copies
    of a news already listed for the user are unranked (rank 0) and not positives.  Asynchronous like top_k."""
    cutoffs = tuple(cutoffs)
    if len(cutoffs) > ops.POOL_RANK_MAX_CUTOFFS or not all(isinstance(c, (int, np.integer)) and c >= 1 for c in cutoffs):
        raise ValueError("cutoffs must be at most %d integers >= 1" % ops.POOL_RANK_MAX_CUTOFFS)
    dev = plan.device
    hist = _histories(plan, hist_news, hist_mask, hist_fresh, hist_life)
    hn, hm = hist[0], hist[1]
    U = hn.shape[0]
    tn = (target_news if torch.is_tensor(target_news) else torch.from_numpy(np.asarray(target_news))).to(dev, torch.int64)
    tm = (target_mask if torch.is_tensor(target_mask) else torch.from_numpy(np.asarray(target_mask))).to(dev, torch.bool)
    if tn.dim() != 2 or tn.shape[0] != U or tm.shape != tn.shape:
        raise ValueError("target_news / target_mask must share one [users, targets] shape")
    if not 1 <= tn.shape[1] <= ops.POOL_RANK_MAX_TARGETS:
        raise ValueError("targets per user must lie in [1, %d]" % ops.POOL_RANK_MAX_TARGETS)
    if tn.numel() and bool(((tn < 0) | (tn >= cache.news_num)).any()):
        raise ValueError("target news ids must lie in [0, %d)" % cache.news_num)
    T = tn.shape[1]
    pos = torch.where(tm, plan.positions(cache.news_num)[tn], -1).to(torch.int32).contiguous()
    columns = ["auc", "mrr", "ndcg5", "ndcg10"] + [n % c for c in cutoffs for n in ("recall@%d", "ndcg@%d")]
    ev = Evaluation(torch.zeros((U, T), dtype=torch.int32, device=dev), torch.zeros(U, dtype=torch.int32, device=dev),
                    torch.zeros(U, dtype=torch.int64, device=dev),
                    torch.empty((U, len(columns)), dtype=torch.float64, device=dev), columns,
                    torch.zeros((), dtype=torch.int64, device=dev))
    with torch.no_grad():
        for u0, u1, s in _scored_batches(model, cache, plan, hist, ev._fallback):
            r = ops.pool_rank_metrics(s, plan.index, pos[u0:u1], cutoffs, plan.news, plan.exclude,
                                      hn[u0:u1] if exclude_clicked else None, hm[u0:u1] if exclude_clicked else None)
            for dst, src in zip((ev.rank, ev.ranked, ev.eligible, ev.metrics), r):
                dst[u0:u1] = src
    return ev
