"""Scoring utilities of the drop-in path (reference util.py:15-129, evaluate.py:32-89).

``compute_scores`` keeps the reference's signature and file outputs; ``evaluate_impressions`` is the
new impression-major entry point it is built on (SURVEY.md §8b "a cached/impression-batched eval is
a new entry point beside compute_scores, returning the same 4-tuple").
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch
import torch.nn as nn

from . import _lib, ops
from .engine import DeviceImpressions
from .synth import Impressions, NewsTable


class RemainingLifetimeWeighting(nn.Module):
    """Remaining-lifetime-guided weighting of the dot-product score (reference util.py:15-49).
    ``forward`` runs lime_click_score_fwd (and its backward when gradients are recorded); the fused
    eval kernels evaluate the same weight inline (score_common.cuh: lifetime_weight)."""

    def __init__(self, config):
        super().__init__()
        self.alpha = config.sigmoid_scaling_alpha
        self.beta = config.penalty_scaling_beta
        self.use_expired_penalty = config.use_expired_penalty
        self.use_remaining_lifetime_weighting = config.use_remaining_lifetime_weighting

    def initialize(self):
        pass

    def forward(self, user_embedding, news_embedding, remaining_lifetime):
        """[B, N, D], [B, N, D], [B, N] -> weighted matching score [B, N] (util.py:23-49)."""
        from . import training
        B, N, D = user_embedding.shape
        return training.click_scores(self, user_embedding.reshape(B * N, D).contiguous(),
                                     news_embedding.reshape(B * N, D).contiguous(), remaining_lifetime, B, N)


@dataclass
class NewsVectorCache:
    """Per-news derived vectors resident in HBM (engine.py docstring for the row layout)."""
    hist_rows: torch.Tensor     # [news_num, 852] fp32
    cand_rows: torch.Tensor     # [news_num, 1720] fp32
    cand16: torch.Tensor = None  # [news_num, 2400] fp16 hi/lo pairs of cand_rows[:, :1200] (tensor-core scoring operand)
    meta: torch.Tensor = None    # [news_num, 8] fp32 per-news scalars of the tensor-core kernel's phase 0
    hist_vg: torch.Tensor = None  # [news_num, 800] fp32: vc | gw of hist_rows interleaved by 4 dims (one 256-bit load per quad)

    @property
    def news_num(self):
        return int(self.hist_rows.shape[0])

    def nbytes(self):
        return self.hist_rows.numel() * 4 + self.cand_rows.numel() * 4 + (self.cand16.numel() * 2 if self.cand16 is not None else 0) + (self.meta.numel() * 4 if self.meta is not None else 0) + (self.hist_vg.numel() * 4 if self.hist_vg is not None else 0)


def build_news_cache(model, news: NewsTable, device=None, chunk=None) -> NewsVectorCache:
    """Encode every news of the corpus once (the reference re-encodes 50 history news per scored
    pair, dataset.py:192-227 + util.py:88-112)."""
    device = device or next(model.parameters()).device
    if chunk is None:       # news per encoder pass: the tensor-core modes amortise their per-launch weight loads over more rows
        eng = model.news_encoder.engine
        chunk = 8192 if (eng.bf16 or eng.x3) else 2048
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a, np.int32)).to(device)
    with torch.no_grad():
        hist, cand = model.scoring.build_rows(t(news.title_text), t(news.body_text), t(news.category),
                                              t(news.subCategory), chunk=chunk)
        cand16 = model.scoring.split_candidates(cand)
        meta = model.scoring.news_meta(hist, cand)
        from .engine import interleave_vg
        hist_vg = interleave_vg(hist)
    return NewsVectorCache(hist, cand, cand16, meta, hist_vg)


def _tail(total_pairs, batch_size):
    """Reference batching (DataLoader(shuffle=False, batch_size), util.py:81): the last
    ``total_pairs % batch_size`` pairs form a short batch whose runtime size drives GraphSAGE."""
    tail_start = (total_pairs // batch_size) * batch_size
    return tail_start, max(1, total_pairs - tail_start)


def score_impressions(model, cache: NewsVectorCache, dimp: DeviceImpressions, batch_size,
                      pair_index_base=0, total_pairs=None, out=None):
    """fp32 scores [P] for every (impression, candidate) pair of ``dimp``; equals what
    compute_scores' loop (util.py:88-112) collects when the reference runs with ``batch_size``."""
    total = dimp.num_pairs if total_pairs is None else total_pairs
    tail_start, prefix_tail = _tail(total, batch_size)
    return model.scoring.score(cache.hist_rows, cache.cand_rows, dimp, prefix_main=batch_size,
                               tail_start=tail_start, prefix_tail=prefix_tail,
                               pair_index_base=pair_index_base, out=out, cand16=cache.cand16, meta=cache.meta, hist_vg=cache.hist_vg)


def evaluate_device(model, cache, dimp, batch_size, pair_index_base=0, total_pairs=None, group=None,
                    scores_out=None, want_ranks=True, sharded=False):
    """The device-side part of evaluate_impressions, fully asynchronous: 3 kernel launches (score,
    rank+metrics, reduce) and -- ONLY when the caller says the impression set is sharded over a process
    group (``group`` given, or ``sharded=True`` for the default group) -- one all-reduce of the five
    partial sums, which every rank of that group must then enter.  A plain call never issues a
    collective: the reference's own distributed flow evaluates on rank 0 alone (trainer.py:342), and an
    implicit all-reduce there would wait for ranks that never call.  Returns device tensors."""
    scores = score_impressions(model, cache, dimp, batch_size, pair_index_base, total_pairs, out=scores_out)
    ranks, per_imp = ops.rank_metrics(scores, dimp.dev["labels"], dimp.dev["cand_off"], want_ranks=want_ranks)
    sums = ops.metrics_reduce(per_imp)
    if group is not None or sharded:
        torch.distributed.all_reduce(sums, group=group)
    return scores, ranks, per_imp, sums


def _means(s):
    """(auc, mrr, ndcg5, ndcg10) from the five sums; NaN when no impression carries both classes of labels
    (an unlabeled test set: the reference returns None there, util.py:124-129)."""
    n = s[4]
    return tuple((x / n) if n > 0 else float("nan") for x in s[:4])


def evaluate_impressions(model, cache, dimp, batch_size, pair_index_base=0, total_pairs=None,
                         group=None, return_details=False, sharded=False):
    """Scores -> per-impression stable ranks -> (auc, mrr, ndcg5, ndcg10) averaged over impressions,
    all on the device.  ``group`` / ``sharded=True``: ``dimp`` is this rank's shard of one impression
    set; the five partial sums are all-reduced (NCCL) and every rank of the group -- all of them must
    call -- returns the global means (SURVEY.md §8e)."""
    scores, ranks, per_imp, sums = evaluate_device(model, cache, dimp, batch_size, pair_index_base,
                                                   total_pairs, group, sharded=sharded)
    s = sums.tolist()                                # device -> host read of the step's result
    result = _means(s)
    if return_details:
        return result, dict(scores=scores, ranks=ranks, per_impression=per_imp, sums=sums)
    return result


def write_rank_file(path, ranks, cand_off):
    """The reference's prediction format (util.py:117-123): line i = '<i+1> [r1,r2,...]', no
    trailing newline."""
    r = ranks.tolist() if torch.is_tensor(ranks) else list(ranks)
    off = cand_off.tolist() if hasattr(cand_off, "tolist") else list(cand_off)
    with open(path, "w", encoding="utf-8") as f:
        for i in range(len(off) - 1):
            f.write(("" if i == 0 else "\n") + str(i + 1) + " " + str(r[off[i]:off[i + 1]]).replace(" ", ""))


def corpus_to_tables(corpus, mode):
    """Adapter from the reference's ``Corpus`` object (corpus.py:361-368, 577-649) to the
    impression-major arrays: consecutive dev/test behaviours with the same impression index are the
    candidates of one impression and share one history."""
    beh = corpus.dev_behaviors if mode == "dev" else corpus.test_behaviors
    indices = np.asarray(corpus.dev_indices if mode == "dev" else corpus.test_indices, np.int64)
    H = corpus.max_history_num
    news = NewsTable(corpus.news_title_text, corpus.news_title_mask, corpus.news_abstract_text,
                     corpus.news_abstract_mask, corpus.news_category, corpus.news_subCategory,
                     int(corpus.config.vocabulary_size), int(corpus.config.category_num),
                     int(corpus.config.subCategory_num))
    n_imp = int(indices[-1]) + 1 if len(indices) else 0
    counts = np.bincount(indices, minlength=n_imp)
    cand_off = np.zeros(n_imp + 1, np.int64)
    np.cumsum(counts, out=cand_off[1:])
    if np.any(np.diff(indices) < 0):
        raise ValueError("behaviours must be grouped by impression (corpus.py:590,636 appends them in order)")
    hist_news = np.zeros((n_imp, H), np.int32)
    hist_mask = np.zeros((n_imp, H), bool)
    hist_fresh = np.zeros((n_imp, H), np.float32)
    hist_life = np.zeros((n_imp, H), np.float32)
    user_id = np.zeros(n_imp, np.int64)

    def pad(lst):                                           # dataset.py:203-205
        v = list(lst)[-H:]
        return np.asarray(v + [0] * max(0, H - len(lst)), np.float32)[:H]

    first = cand_off[:-1]
    for i in range(n_imp):
        if counts[i] == 0:
            continue
        b = beh[first[i]]
        user_id[i] = b[0]
        hist_news[i] = np.asarray(b[1], np.int32)
        hist_mask[i] = np.asarray(b[2], bool)
        hist_fresh[i] = pad(b[7])
        hist_life[i] = pad(b[8])
    cand_news = np.asarray([b[3] for b in beh], np.int32)
    cand_fresh = np.asarray([b[5] for b in beh], np.float32)
    cand_life = np.asarray([b[6] for b in beh], np.float32)
    imp = Impressions(hist_news, hist_mask, hist_fresh, hist_life, cand_off, cand_news, cand_fresh,
                      cand_life, np.zeros(len(beh), np.uint8), user_id)
    return news, imp


def _read_truth(path, cand_off):
    """Labels from the reference's truth file ('<impr> [l1,l2,...]', config.py:262-276)."""
    import json
    labels = np.zeros(int(cand_off[-1]), np.uint8)
    with open(path, "r", encoding="utf-8") as f:
        for i, line in enumerate(f):
            _, arr = line.strip("\n").split()
            arr = json.loads(arr)
            labels[cand_off[i]:cand_off[i] + len(arr)] = arr
    return labels


def remaining_lifetime(config, cand_fresh, cand_category):
    """Remaining lifetime handed to RemainingLifetimeWeighting per candidate (util.py:98-104): fp32 [P] for
    lifetime_type 'fixed' (fixed_lifetime - freshness) and 'topic_wise' (category_lifetime_map[category] - freshness),
    None for 'user_topic' (the scoring kernel then uses lifetime - freshness).  cand_fresh: fp32 numpy [P];
    cand_category: a callable returning the candidates' category ids (evaluated for 'topic_wise' only)."""
    if config.lifetime_type == "fixed":                                     # util.py:98-99
        return np.float32(config.fixed_lifetime) - cand_fresh
    if config.lifetime_type == "topic_wise":                                # util.py:100-102
        clm = config.category_lifetime_map
        clm = clm.detach().cpu().numpy() if torch.is_tensor(clm) else np.asarray(clm)
        return clm[cand_category()].astype(np.float32) - cand_fresh
    if config.lifetime_type != "user_topic":
        raise ValueError("Invalid lifetime_type")
    return None


def compute_scores(model, corpus, batch_size, mode, result_file, dataset):
    """Reference signature (util.py:77).  Builds the news-vector cache, scores every dev/test pair
    with the fused kernel, writes the rank file in the reference's format and returns
    (auc, mrr, ndcg5, ndcg10) against ``<mode>/ref/truth-<dataset>.txt`` (None x4 for the unlabeled
    MIND-large test set, util.py:124-129)."""
    assert mode in ["dev", "test"], "mode must be chosen from 'dev' or 'test'"
    config = model.config
    news, imp = corpus_to_tables(corpus, mode)
    device = next(model.parameters()).device
    model.eval()
    remaining = remaining_lifetime(config, imp.cand_fresh, lambda: news.category[imp.cand_news])
    labeled = dataset != "large" or mode != "test"
    if labeled:
        imp.labels = _read_truth(mode + "/ref/truth-%s.txt" % dataset, imp.cand_off)
    with torch.no_grad():
        cache = build_news_cache(model, news, device)
        dimp = DeviceImpressions(imp, device, cand_remaining=remaining, num_buckets=config.num_buckets)
        # never a collective here: the reference calls compute_scores on rank 0 only (trainer.py:342)
        metrics, det = evaluate_impressions(model, cache, dimp, batch_size, return_details=True)
    write_rank_file(result_file, det["ranks"].cpu(), imp.cand_off)
    if labeled:
        return metrics
    return None, None, None, None            # unlabeled MIND-large test set: prediction file only (util.py:124-129)
