"""Scoring utilities of the drop-in path (reference util.py:15-129, evaluate.py:32-89).

``compute_scores`` keeps the reference's signature and file outputs; ``evaluate_impressions`` is the
new impression-major entry point it is built on (SURVEY.md §8b "a cached/impression-batched eval is
a new entry point beside compute_scores, returning the same 4-tuple").
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np
import torch
import torch.nn as nn

from . import _lib, ops
from .engine import CAND_LD, D, HIST_LD, TAB_REPLICAS, DeviceImpressions, _fingerprint
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
    """Per-news derived vectors resident in HBM (engine.py docstring for the row layout).

    The five arrays are views of buffers with room for ``capacity`` rows (DESIGN.md section 2b), so that
    extend_news_cache can append news in place; cand16 is followed by its bucket-pair tail, which always
    starts right after the live rows.  ``fingerprint``: the ScoringEngine fold fingerprint of the build."""
    hist_rows: torch.Tensor     # [news_num, 852] fp32
    cand_rows: torch.Tensor     # [news_num, 1720] fp32
    cand16: torch.Tensor = None  # [news_num + tail, 2400] fp16 hi/lo pairs of cand_rows[:, :1200], then the bucket-pair rows (tensor-core scoring operand)
    meta: torch.Tensor = None    # [news_num, 8] fp32 per-news scalars of the tensor-core kernel's phase 0
    hist_vg: torch.Tensor = None  # [news_num, 800] fp32: vc | gw of hist_rows interleaved by 4 dims (one 256-bit load per quad)
    fingerprint: tuple = field(default=None, repr=False)
    buffers: tuple = field(default=None, repr=False)    # (hist, cand, cand16, meta, hist_vg) with capacity rows (+ the tail)

    @property
    def news_num(self):
        return int(self.hist_rows.shape[0])

    @property
    def capacity(self):
        return int(self.buffers[0].shape[0]) if self.buffers is not None else self.news_num

    def capacity_nbytes(self):
        """Bytes the buffers hold, headroom included (nbytes counts the live rows only)."""
        if self.buffers is None:
            return self.nbytes()
        return sum(b.numel() * b.element_size() for b in self.buffers)

    def nbytes(self):
        return self.hist_rows.numel() * 4 + self.cand_rows.numel() * 4 + (self.cand16.numel() * 2 if self.cand16 is not None else 0) + (self.meta.numel() * 4 if self.meta is not None else 0) + (self.hist_vg.numel() * 4 if self.hist_vg is not None else 0)

    def _set_rows(self, n, tail):
        """Point the five arrays at the first n rows of the buffers; cand16 with its tail (rewritten by the caller)."""
        H, C, C16, M, VG = self.buffers
        self.hist_rows, self.cand_rows, self.meta, self.hist_vg = H[:n], C[:n], M[:n], VG[:n]
        self.cand16 = C16[:n + tail]


def _chunk(model):
    """News per encoder pass: the tensor-core modes amortise their per-launch weight loads over more rows."""
    eng = model.news_encoder.engine
    return 8192 if (eng.bf16 or eng.x3) else 2048


def _write_tail(model, cache):
    """TAB_REPLICAS copies of the bucket-pair rows (ctab16) right after the live rows of cand16."""
    ctab16 = model.scoring.fold()["ctab16"]
    nb2, n = ctab16.shape[0], cache.news_num
    cache.cand16[n:].view(TAB_REPLICAS, nb2, 2400).copy_(ctab16.unsqueeze(0).expand(TAB_REPLICAS, nb2, 2400))


def build_news_cache(model, news: NewsTable, device=None, chunk=None, capacity=None) -> NewsVectorCache:
    """Encode every news of the corpus once (the reference re-encodes 50 history news per scored
    pair, dataset.py:192-227 + util.py:88-112).  ``capacity``: rows to allocate (at least news_num; default
    news_num + max(news_num / 8, 1024)), the room extend_news_cache fills before it reallocates; capacity=news_num
    allocates no headroom (cache.capacity_nbytes() reports what the buffers hold)."""
    device = device or next(model.parameters()).device
    chunk = chunk or _chunk(model)
    N = news.news_num
    cap = max(N, N + max(N // 8, 1024) if capacity is None else int(capacity))
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a, np.int32)).to(device)
    se = model.scoring
    with torch.no_grad():
        tail = TAB_REPLICAS * se.fold()["ctab16"].shape[0]
        f32 = dict(dtype=torch.float32, device=device)
        cache = NewsVectorCache(None, None, buffers=(
            torch.empty(cap, HIST_LD, **f32), torch.empty(cap, CAND_LD, **f32),
            torch.empty(cap + tail, 2400, dtype=torch.float16, device=device),
            torch.empty(cap, 8, **f32), torch.empty(cap, 2 * D, **f32)))
        cache._set_rows(N, tail)
        # the rows are built in place and the kernel derives the other roles from them (destination = source row)
        se.build_rows(t(news.title_text), t(news.body_text), t(news.category), t(news.subCategory), chunk=chunk,
                      out=(cache.hist_rows, cache.cand_rows), host_topics=(news.category, news.subCategory))
        cache.fingerprint = se._fp
        ops.cache_write_rows(cache.hist_rows, cache.cand_rows, torch.arange(N, device=device), cache.hist_rows,
                             cache.cand_rows, cache.cand16, cache.meta, cache.hist_vg)
        _write_tail(model, cache)
    return cache


def table_sizes(model):
    """(vocabulary size, category ids, subCategory ids) the model's embedding tables accept."""
    lime, base = model.news_encoder, model.news_encoder.base_news_encoder
    return (int(base.word_embedding.weight.shape[0]),
            min(int(lime.category_embedding.weight.shape[0]), int(base.category_embedding.weight.shape[0])),
            min(int(lime.subCategory_embedding.weight.shape[0]), int(base.subCategory_embedding.weight.shape[0])))


def validate_news(news: NewsTable, vocabulary_size, category_num, subCategory_num):
    """Host-side checks of news to encode into a cache: [n, 32] titles and [n, 128] bodies, [n] category and
    subCategory, every id inside the model's tables.  -> (title, body, category, subCategory) int32 numpy arrays."""
    title, body = np.asarray(news.title_text), np.asarray(news.body_text)
    cat, sub = np.asarray(news.category), np.asarray(news.subCategory)
    if title.ndim != 2 or title.shape[1] != 32 or body.ndim != 2 or body.shape[1] != 128:
        raise ValueError("news titles must be [n, 32] and bodies [n, 128] (got %s, %s)" % (title.shape, body.shape))
    n = title.shape[0]
    if body.shape[0] != n or cat.shape != (n,) or sub.shape != (n,):
        raise ValueError("titles, bodies, category and subCategory must describe the same %d news" % n)
    for a, name in ((title, "title"), (body, "body"), (cat, "category"), (sub, "subCategory")):
        if not np.issubdtype(a.dtype, np.integer):
            raise ValueError("%s ids must be integers (got %s)" % (name, a.dtype))
    for a, hi, name in ((title, vocabulary_size, "word"), (body, vocabulary_size, "word"),
                        (cat, category_num, "category"), (sub, subCategory_num, "subCategory")):
        if a.size and (a.min() < 0 or a.max() >= hi):
            raise ValueError("%s ids must lie in [0, %d)" % (name, hi))
    return tuple(np.ascontiguousarray(a, np.int32) for a in (title, body, cat, sub))


def validate_refresh_rows(rows, news_num, n):
    """Host-side checks of the rows refresh_news_cache re-encodes: n ids in [1, news_num), each at most once (row 0 is
    the pad news).  -> int64 numpy array."""
    r = rows.detach().cpu().numpy() if torch.is_tensor(rows) else np.asarray(rows)
    if r.ndim != 1 or r.shape[0] != n:
        raise ValueError("rows must be a 1-D array with one cache row per news (%d)" % n)
    if r.size and not np.issubdtype(r.dtype, np.integer):
        raise ValueError("rows must be integer cache row ids")
    r = r.astype(np.int64)
    if r.size and (r.min() < 1 or r.max() >= news_num):
        raise ValueError("rows must lie in [1, %d): row 0 is the pad news" % news_num)
    if np.unique(r).size != r.size:
        raise ValueError("rows must not repeat a cache row")
    return r


def _check_weights(model, cache):
    if cache.fingerprint is None or cache.buffers is None:
        raise ValueError("the cache was not made by build_news_cache")
    if _fingerprint(model.scoring._params()) != cache.fingerprint:
        raise ValueError("the model's weights changed since the cache was built: rebuild it with build_news_cache")


def _encode(model, cache, arrays):
    """validate_news' arrays -> freshly built (hist, cand) rows with topic ids stamped, or None for n = 0."""
    title, body, cat, sub = arrays
    if title.shape[0] == 0:
        return None
    dev = cache.hist_rows.device
    t = lambda a: torch.from_numpy(a).to(dev)
    return model.scoring.build_rows(t(title), t(body), t(cat), t(sub), chunk=_chunk(model), host_topics=(cat, sub))


def extend_news_cache(model, cache: NewsVectorCache, news: NewsTable) -> torch.Tensor:
    """Encode ``news`` (new news only, no pad row) and append them to ``cache`` in place.  -> their cache row ids,
    int64 [n] on the device (what recommend.plan takes).  The arrays grow inside the buffers' capacity; past it every
    buffer is reallocated 1.5 times larger and the live rows are copied over.  Asynchronous on the current stream
    apart from the host-side checks; raises ValueError for bad ids or shapes and when the model's weights changed since
    the build."""
    _check_weights(model, cache)
    arrays = validate_news(news, *table_sizes(model))
    n0, n = cache.news_num, arrays[0].shape[0]
    tail = cache.cand16.shape[0] - n0
    if n0 + n + tail >= 2 ** 31:          # news_num and the cand16 tensor map count rows in int32
        raise ValueError("a cache holds fewer than 2^31 rows")
    with torch.no_grad():
        rows = _encode(model, cache, arrays)
        dev = cache.hist_rows.device
        if rows is None:
            return torch.zeros(0, dtype=torch.int64, device=dev)
        if n0 + n > cache.capacity:
            cap = min(max(n0 + n, cache.capacity + cache.capacity // 2), 2 ** 31 - 1 - tail)
            old = (cache.hist_rows, cache.cand_rows, cache.cand16[:n0], cache.meta, cache.hist_vg)
            cache.buffers = tuple(torch.empty((cap + (tail if i == 2 else 0),) + tuple(a.shape[1:]), dtype=a.dtype, device=dev)
                                  for i, a in enumerate(old))
            for b, a in zip(cache.buffers, old):
                b[:n0].copy_(a)
            del old
        cache._set_rows(n0 + n, tail)
        ids = torch.arange(n0, n0 + n, device=dev)
        ops.cache_write_rows(rows[0], rows[1], ids, cache.hist_rows, cache.cand_rows, cache.cand16, cache.meta, cache.hist_vg)
        _write_tail(model, cache)
    return ids


def refresh_news_cache(model, cache: NewsVectorCache, rows, news: NewsTable):
    """Re-encode existing cache rows in place (edited news): ``rows`` [n] ids in [1, news_num), each at most once, row i
    becomes the encoding of news i of ``news``.  Plans made before keep scoring correctly with the new rows; re-plan a
    pool whose news changed category, or its sort order (hence its work units) is stale.  Asynchronous and checked like
    extend_news_cache."""
    _check_weights(model, cache)
    arrays = validate_news(news, *table_sizes(model))
    r = validate_refresh_rows(rows, cache.news_num, arrays[0].shape[0])
    with torch.no_grad():
        built = _encode(model, cache, arrays)
        if built is None:
            return
        dst = torch.from_numpy(r).to(cache.hist_rows.device)
        ops.cache_write_rows(built[0], built[1], dst, cache.hist_rows, cache.cand_rows, cache.cand16, cache.meta, cache.hist_vg)


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
