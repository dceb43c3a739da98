"""Full-pool ranking evaluation on the GPU: lime_pool_rank_metrics against a NumPy reference (exact ranks and counts,
metrics to 1e-12), against lime_rank_metrics and lime_pool_topk on the same scores, and recommend.evaluate against the
materialised impression set (every user one impression whose candidates are the pool in the caller's order)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import lime_cikm25_b200 as L  # noqa: E402
from lime_cikm25_b200 import engine, ops, recommend, synth, util  # noqa: E402
from oracle.ref_import import make_config  # noqa: E402

DEV = "cuda"
CUTOFFS = (1, 3, 10, 100, 5000, 400000)          # K > C for every pool below but the largest


def make_scores(U, C, dist, rng):
    if dist == "random":
        return rng.standard_normal((U, C)).astype(np.float32)
    if dist == "ties":
        return (rng.integers(-2, 3, (U, C)) * 0.5).astype(np.float32)
    vals = np.asarray([-0.0, 0.0, np.nan, 1.5, -1.5, np.inf, -np.inf], np.float32)     # signed zeros, NaN, infinities
    return vals[rng.integers(0, vals.size, (U, C))]


def eligible_mask(scores, pool_news=None, exclude=None, hist_news=None, hist_mask=None):
    ok = ~np.isnan(scores)
    if exclude is not None:
        ok &= (exclude == 0)[None, :]
    if hist_news is not None:
        for u in range(scores.shape[0]):
            ok[u] &= ~np.isin(pool_news, hist_news[u][hist_mask[u] != 0])
    return ok


def ref_order(scores_u, ok_u, pool_index):
    """Eligible positions of one user in top_k's order: score descending (-0.0 == +0.0), then ascending pool_index."""
    pos = np.nonzero(ok_u)[0]
    return pos[np.lexsort((pool_index[pos], -scores_u[pos]))]


def ref_metrics(r, N, cutoffs):
    """fp64 metrics row of ranks r (1-based) among N eligible positions."""
    n = r.size
    row = np.full(4 + 2 * len(cutoffs), np.nan)
    if n == 0:
        return row
    g = 1.0 / np.log2(r + 1.0)
    ideal = lambda K: float(np.sum(1.0 / np.log2(np.arange(1, min(n, K) + 1) + 1.0)))
    with np.errstate(invalid="ignore", divide="ignore"):
        row[0] = np.float64(int(np.sum(N - r.astype(np.int64))) - n * (n - 1) // 2) / (np.float64(n) * np.float64(N - n))
    row[1] = np.mean(1.0 / r)
    row[2] = g[r <= 5].sum() / ideal(5)
    row[3] = g[r <= 10].sum() / ideal(10)
    for q, K in enumerate(cutoffs):
        row[4 + 2 * q] = np.sum(r <= K) / n
        row[5 + 2 * q] = g[r <= K].sum() / ideal(K)
    return row


def ref_rank(scores, pool_index, target_pos, cutoffs, pool_news=None, exclude=None, hist_news=None, hist_mask=None):
    U, C = scores.shape
    T = target_pos.shape[1]
    ok = eligible_mask(scores, pool_news, exclude, hist_news, hist_mask)
    rank = np.zeros((U, T), np.int64)
    ranked = np.zeros(U, np.int64)
    eligible = ok.sum(1)
    metrics = np.zeros((U, 4 + 2 * len(cutoffs)))
    for u in range(U):
        pos_rank = np.zeros(C, np.int64)
        pos_rank[ref_order(scores[u], ok[u], pool_index)] = np.arange(1, eligible[u] + 1)
        seen = set()
        for t, p in enumerate(target_pos[u]):
            if 0 <= p < C and ok[u, p] and p not in seen:
                rank[u, t] = pos_rank[p]
                seen.add(p)
        r = rank[u][rank[u] > 0]
        ranked[u] = r.size
        metrics[u] = ref_metrics(r.astype(np.float64), int(eligible[u]), cutoffs)
    return rank, ranked, eligible, metrics


def make_targets(scores, T, rng, pool_index, pool_news=None, exclude=None, hist_news=None, hist_mask=None):
    """Random pool positions plus every unranked kind: duplicates, -1 slots, excluded, clicked and NaN-scored positions;
    user 0 holds the T best eligible positions, user 1 the T worst."""
    U, C = scores.shape
    tp = rng.integers(0, C, (U, T)).astype(np.int32)
    ok = eligible_mask(scores, pool_news, exclude, hist_news, hist_mask)
    for u in range(U):
        special = []
        if T >= 2:
            special += [("dup", 1), ("none", 2)]
        for kind, slot in special:
            if slot < T:
                tp[u, slot] = tp[u, 0] if kind == "dup" else -1
        extra = 3
        for bad in (np.isnan(scores[u]), None if exclude is None else exclude != 0,
                    None if hist_news is None else np.isin(pool_news, hist_news[u][hist_mask[u] != 0])):
            if bad is not None and bad.any() and extra < T:
                tp[u, extra] = rng.choice(np.nonzero(bad)[0])
                extra += 1
    for u, part in ((0, slice(None, T)), (1, slice(-T, None))):
        if u < U:
            order = ref_order(scores[u], ok[u], pool_index)[part]
            tp[u] = -1
            tp[u, :order.size] = order
    return tp


def run_kernel(scores, pool_index, target_pos, cutoffs, pool_news=None, exclude=None, hist_news=None, hist_mask=None):
    t = lambda a, dt: None if a is None else torch.as_tensor(a).to(DEV, dt).contiguous()
    out = ops.pool_rank_metrics(t(scores, torch.float32), t(pool_index, torch.int32), t(target_pos, torch.int32), cutoffs,
                                t(pool_news, torch.int32), t(exclude, torch.uint8), t(hist_news, torch.int32),
                                t(hist_mask, torch.uint8))
    return tuple(x.cpu().numpy() for x in out)


def check(got, want):
    gr, gn, ge, gm = got
    wr, wn, we, wm = want
    assert np.array_equal(gn, wn)
    assert np.array_equal(ge, we)
    assert np.array_equal(gr, wr)
    np.testing.assert_allclose(gm, wm, rtol=0, atol=1e-12, equal_nan=True)


def world_pool(U, C, dist, H, rng):
    scores = make_scores(U, C, dist, rng)
    pool_index = rng.permutation(C).astype(np.int32)
    pool_news = rng.permutation(np.arange(1, C + 1)).astype(np.int32)
    exclude = (rng.random(C) < 0.1).astype(np.uint8)
    hist_news = rng.integers(1, 2 * C + 1, (U, H)).astype(np.int32)
    hist_mask = rng.random((U, H)) < 0.7
    return scores, pool_index, pool_news, exclude, hist_news, hist_mask


# ---- kernel ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("U,C,T", [(1, 1, 1), (3, 37, 5), (5, 4097, 64), (2, 300000, 256), (64, 65238, 8)])
@pytest.mark.parametrize("dist", ["random", "ties", "special"])
@pytest.mark.parametrize("excl", [False, True])
def test_pool_rank_matches_reference(lib, U, C, T, dist, excl):
    rng = np.random.default_rng(U * 11 + C + T)
    scores, pool_index, pool_news, exclude, hist_news, hist_mask = world_pool(U, C, dist, 20, rng)
    kw = dict(pool_news=pool_news, exclude=exclude, hist_news=hist_news, hist_mask=hist_mask) if excl else {}
    tp = make_targets(scores, T, rng, pool_index, **kw)
    check(run_kernel(scores, pool_index, tp, CUTOFFS, **kw), ref_rank(scores, pool_index, tp, CUTOFFS, **kw))


def test_pool_rank_edge_rows(lib):
    """No ranked target -> NaN row; every eligible position a target (N == n) -> AUC NaN; nothing eligible."""
    C = 6
    scores = np.asarray([[3, 2, 1, 0, -1, -2], [3, 2, 1, 0, -1, -2], [np.nan] * 6], np.float32)
    pool_index = np.arange(C, dtype=np.int32)
    exclude = np.asarray([0, 0, 1, 1, 1, 1], np.uint8)
    tp = np.asarray([[-1, 5, 4], [1, 0, 0], [0, 1, 2]], np.int32)
    got = run_kernel(scores, pool_index, tp, (1, 2), exclude=exclude)
    check(got, ref_rank(scores, pool_index, tp, (1, 2), exclude=exclude))
    rank, ranked, eligible, m = got
    assert np.isnan(m[0]).all() and ranked[0] == 0 and eligible[0] == 2
    assert list(rank[1]) == [2, 1, 0] and np.isnan(m[1, 0]) and m[1, 1] == 0.75
    assert np.isnan(m[2]).all() and eligible[2] == 0


@pytest.mark.parametrize("U,C,T,dist", [(3, 37, 5, "ties"), (5, 4097, 64, "random"), (4, 4097, 64, "special")])
def test_pool_rank_matches_rank_metrics(lib, U, C, T, dist):
    """Each user's eligible positions in caller order form one impression labelled by the targets: lime_rank_metrics
    gives the same ranks and the same four metrics."""
    rng = np.random.default_rng(C + T)
    scores, pool_index, pool_news, exclude, hist_news, hist_mask = world_pool(U, C, dist, 20, rng)
    kw = dict(pool_news=pool_news, exclude=exclude, hist_news=hist_news, hist_mask=hist_mask)
    tp = make_targets(scores, T, rng, pool_index, **kw)
    rank, ranked, eligible, m = run_kernel(scores, pool_index, tp, (10,), **kw)
    ok = eligible_mask(scores, **kw)
    by_caller = np.argsort(pool_index)
    flat_s, flat_y, off, where = [], [], [0], []
    for u in range(U):
        pos = by_caller[ok[u, by_caller]]
        y = np.isin(pos, tp[u][rank[u] > 0])
        where.append({p: off[-1] + i for i, p in enumerate(pos)})
        flat_s.append(scores[u, pos])
        flat_y.append(y.astype(np.uint8))
        off.append(off[-1] + pos.size)
    t = lambda a, dt: torch.as_tensor(np.concatenate(a) if isinstance(a, list) else a).to(DEV, dt).contiguous()
    r2, m2 = ops.rank_metrics(t(flat_s, torch.float32), t(flat_y, torch.uint8), t(np.asarray(off), torch.int64))
    r2 = r2.cpu().numpy()
    for u in range(U):
        assert eligible[u] == off[u + 1] - off[u]
        for s, p in enumerate(tp[u]):
            if rank[u, s] > 0:
                assert rank[u, s] == r2[where[u][p]], (u, s)
    np.testing.assert_allclose(m[:, :4], m2.cpu().numpy(), rtol=0, atol=1e-12, equal_nan=True)


@pytest.mark.parametrize("U,C,T,k,dist", [(3, 37, 5, 37, "ties"), (4, 1000, 64, 1000, "special"), (3, 65238, 64, 100, "random")])
def test_pool_rank_matches_pool_topk(lib, U, C, T, k, dist):
    """Rank r <= k means pool_topk(k) returns the target at position r; targets ranked beyond k are not returned."""
    rng = np.random.default_rng(C + k)
    scores, pool_index, pool_news, exclude, hist_news, hist_mask = world_pool(U, C, dist, 20, rng)
    kw = dict(pool_news=pool_news, exclude=exclude, hist_news=hist_news, hist_mask=hist_mask)
    tp = make_targets(scores, T, rng, pool_index, **kw)
    rank, ranked, eligible, _ = run_kernel(scores, pool_index, tp, (), **kw)
    t = lambda a, dt: torch.as_tensor(a).to(DEV, dt).contiguous()
    idx, _, cnt = ops.pool_topk(t(scores, torch.float32), k, t(pool_index, torch.int32), t(pool_news, torch.int32),
                                t(exclude, torch.uint8), t(hist_news, torch.int32), t(hist_mask, torch.uint8))
    idx, cnt = idx.cpu().numpy(), cnt.cpu().numpy()
    for u in range(U):
        for s, p in enumerate(tp[u]):
            r = rank[u, s]
            if 0 < r <= k:
                assert idx[u, r - 1] == pool_index[p], (u, s, r)
            elif r > k:
                assert pool_index[p] not in idx[u, :cnt[u]], (u, s, r)
        if k == C:
            assert eligible[u] == cnt[u]


def test_pool_rank_rejects_bad_arguments(lib):
    import ctypes
    s = torch.zeros(2, 8, device=DEV)
    pi = torch.arange(8, dtype=torch.int32, device=DEV)
    tp = torch.zeros(2, 4, dtype=torch.int32, device=DEV)
    for T in (0, 257):
        with pytest.raises(L._lib.LimeError, match="targets="):
            ops.pool_rank_metrics(s, pi, torch.zeros(2, T, dtype=torch.int32, device=DEV))
    with pytest.raises(L._lib.LimeError, match="num_cutoffs="):
        ops.pool_rank_metrics(s, pi, tp, tuple(range(1, 10)))
    with pytest.raises(L._lib.LimeError, match="cutoff"):
        ops.pool_rank_metrics(s, pi, tp, (10, 0))
    hn = torch.zeros(2, 225, dtype=torch.int32, device=DEV)
    with pytest.raises(L._lib.LimeError, match="max_history="):
        ops.pool_rank_metrics(s, pi, tp, (), pi, None, hn, torch.ones(2, 225, dtype=torch.uint8, device=DEV))
    o = torch.empty(64, dtype=torch.float64, device=DEV)
    sc = torch.empty(1024, dtype=torch.uint8, device=DEV)
    cut = (ctypes.c_int32 * 1)(10)
    args = lambda **kw: [kw.get("scores", s.data_ptr()), 2, kw.get("pool", 8), kw.get("pi", pi.data_ptr()), None, None, None,
                         None, 0, tp.data_ptr(), 4, cut, 1, o.data_ptr(), o.data_ptr(), o.data_ptr(), o.data_ptr(),
                         kw.get("scratch", sc.data_ptr()), None]
    assert lib.lime_pool_rank_metrics(*args()) == 0
    torch.cuda.synchronize()
    for bad in (dict(scores=None), dict(pi=None), dict(scratch=None)):
        assert lib.lime_pool_rank_metrics(*args(**bad)) != 0 and b"null" in lib.lime_last_error()
    assert lib.lime_pool_rank_metrics(*args(pool=1 << 31)) != 0 and b"pool" in lib.lime_last_error()
    assert lib.lime_pool_rank_scratch_bytes(2, 4) == 2 * 9 * 4 and lib.lime_pool_rank_scratch_bytes(2, 257) == 0


# ---- end to end ----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def world(lib):
    cfg = make_config(vocabulary_size=5000, batch_size=32, word_embedding_init="skip")
    model = L.Model(cfg)
    model.initialize()
    synth.synthetic_parameters(model, 7)
    model = model.to(DEV).eval()
    news = synth.make_news_table(3000, vocabulary_size=5000, seed=11)
    with torch.no_grad():
        cache = util.build_news_cache(model, news)
    rng = np.random.default_rng(5)
    C = 700
    pool_news = rng.choice(np.arange(1, news.news_num), C, replace=False).astype(np.int32)
    pool_fresh = np.exp(rng.uniform(np.log(60.0), np.log(3e5), C)).astype(np.float32)
    pool_life = np.exp(rng.uniform(np.log(3600.0), np.log(6e5), C)).astype(np.float32)
    exclude = (rng.random(C) < 0.1).astype(np.uint8)
    imp = synth.make_impressions(40, news.news_num, cand_fixed=2, seed=6)
    imp.hist_news[1, :5] = pool_news[:5]                                   # clicked pool news
    imp.hist_mask[1, :5] = True
    imp.hist_mask[2] = False                                               # an empty history
    U, T = imp.num_impressions, 8
    tn = pool_news[rng.integers(0, C, (U, T))].astype(np.int64)
    tm = rng.random((U, T)) < 0.9
    outside = np.setdiff1d(np.arange(1, news.news_num), pool_news)
    kept = np.nonzero(exclude == 0)[0]
    tn[0, :4] = outside[0], pool_news[np.nonzero(exclude)[0][0]], pool_news[1], pool_news[1]
    tm[0, :4] = True, True, False, True                # outside the pool, excluded, a masked slot, its news listed again
    tn[1, 1], tm[1, 1] = pool_news[kept[kept < 5][0]], True                # a clicked news
    dup = next(j for j in kept if pool_news[j] not in tn[2, :4])
    tn[2, 4] = tn[2, 5] = pool_news[dup]                                   # a duplicate (user 2: empty history)
    tm[2, 4] = tm[2, 5] = True
    tn[3], tm[3] = outside[:T], True                                       # no ranked target
    return dict(cfg=cfg, model=model, news=news, cache=cache, pool=(pool_news, pool_fresh, pool_life), exclude=exclude,
                imp=imp, targets=(tn, tm))


def materialised(world, pool, remaining=None):
    """Every user one impression whose candidates are the pool in the caller's order -> scores [U, C] (the reference's
    full mini-batch prefix)."""
    imp, model = world["imp"], world["model"]
    pn, pf, pl = pool
    U, C = imp.num_impressions, pn.size
    m = synth.Impressions(imp.hist_news, imp.hist_mask, imp.hist_fresh, imp.hist_life, np.arange(U + 1, dtype=np.int64) * C,
                          np.tile(pn, U), np.tile(pf, U), np.tile(pl, U), np.zeros(U * C, np.uint8), imp.user_id)
    d = engine.DeviceImpressions(m, DEV, cand_remaining=None if remaining is None else np.tile(remaining, U),
                                 num_buckets=world["cfg"].num_buckets)
    c = world["cache"]
    with torch.no_grad():
        s = model.scoring.score(c.hist_rows, c.cand_rows, d, prefix_main=world["cfg"].batch_size, cand16=c.cand16, meta=c.meta,
                                hist_vg=c.hist_vg)
    return s.view(U, C).cpu().numpy().copy()


def run_evaluate(world, pool=None, cutoffs=(1, 10, 50, 1000), **kw):
    imp = world["imp"]
    with torch.no_grad():
        plan = recommend.plan(world["model"], world["cache"], *(pool or world["pool"]), exclude=world["exclude"])
        return recommend.evaluate(world["model"], world["cache"], plan, imp.hist_news, imp.hist_mask, imp.hist_fresh,
                                  imp.hist_life, *world["targets"], cutoffs=cutoffs, **kw)


def host(ev):
    return [x.cpu().numpy() for x in (ev.rank, ev.ranked, ev.eligible, ev.metrics)]


@pytest.fixture
def exact_mode():
    ops.score_configure(ops.SCORE_EXACT)
    yield
    ops.score_configure(ops.SCORE_AUTO)


@pytest.mark.parametrize("exclude_clicked,lifetime", [(True, None), (False, None), (True, "fixed"), (True, "topic_wise")])
def test_evaluate_exact_mode_matches_materialised(world, exact_mode, exclude_clicked, lifetime):
    """Ranks and metrics of recommend.evaluate = lime_rank_metrics on the materialised set, restricted to the eligible
    positions and labelled by the ranked targets."""
    cfg, news, imp = world["model"].config, world["news"], world["imp"]
    pn, pf, _ = world["pool"]
    tn, tm = world["targets"]
    cutoffs = (1, 10, 50, 1000)
    saved = cfg.lifetime_type, cfg.category_lifetime_map
    if lifetime is not None:
        cfg.lifetime_type = lifetime
        cfg.category_lifetime_map = torch.linspace(3600.0, 2e5, news.category_num)
    try:
        remaining = None if lifetime is None else util.remaining_lifetime(cfg, pf, lambda: news.category[pn])
        s = materialised(world, world["pool"], remaining=remaining)
        ev = run_evaluate(world, cutoffs=cutoffs, exclude_clicked=exclude_clicked)
        rank, ranked, eligible, m = host(ev)
    finally:
        cfg.lifetime_type, cfg.category_lifetime_map = saved
    U, C = s.shape
    flat_s, flat_y, off, want_rank = [], [], [0], np.zeros_like(rank)
    for u in range(U):
        ok = ~np.isnan(s[u]) & (world["exclude"] == 0)
        if exclude_clicked:
            ok &= ~np.isin(pn, imp.hist_news[u][imp.hist_mask[u]])
        pos = np.nonzero(ok)[0]
        seen, y = set(), np.zeros(pos.size, np.uint8)
        for t in range(tn.shape[1]):
            hit = np.nonzero(pn[pos] == tn[u, t])[0]
            if tm[u, t] and hit.size and tn[u, t] not in seen:
                seen.add(tn[u, t])
                y[hit[0]] = 1
                want_rank[u, t] = -(off[-1] + hit[0]) - 1               # resolved below from lime_rank_metrics' ranks
        flat_s.append(s[u, pos])
        flat_y.append(y)
        off.append(off[-1] + pos.size)
    t = lambda a, dt: torch.as_tensor(np.concatenate(a) if isinstance(a, list) else a).to(DEV, dt).contiguous()
    r2, m2 = ops.rank_metrics(t(flat_s, torch.float32), t(flat_y, torch.uint8), t(np.asarray(off), torch.int64))
    r2, m2 = r2.cpu().numpy(), m2.cpu().numpy()
    want_rank = np.where(want_rank < 0, r2[np.maximum(-want_rank - 1, 0)], 0)
    assert np.array_equal(rank, want_rank)
    assert np.array_equal(eligible, np.diff(off))
    assert np.array_equal(ranked, (rank > 0).sum(1))
    np.testing.assert_allclose(m[:, :4], m2, rtol=0, atol=1e-12, equal_nan=True)
    for u in range(U):
        r = rank[u][rank[u] > 0].astype(np.float64)
        np.testing.assert_allclose(m[u], ref_metrics(r, int(eligible[u]), cutoffs), rtol=0, atol=1e-12, equal_nan=True)
    assert rank[0, 0] == 0 and rank[0, 1] == 0 and rank[0, 2] == 0               # outside, excluded, masked
    assert (rank[0, 3] > 0) == (world["exclude"][1] == 0)                         # the copy after a masked slot counts
    assert (rank[1, 1] == 0) == exclude_clicked                                   # clicked
    assert rank[2, 4] > 0 and rank[2, 5] == 0                                     # the second copy is unranked
    assert ranked[3] == 0 and np.isnan(m[3]).all()
    means = ev.means()
    keep = ranked > 0
    assert means["users"] == keep.sum() and ev.columns[4:] == ["recall@1", "ndcg@1", "recall@10", "ndcg@10", "recall@50",
                                                                 "ndcg@50", "recall@1000", "ndcg@1000"]
    for i, c in enumerate(ev.columns):
        assert means[c] == pytest.approx(float(m[keep, i].mean()), nan_ok=True)


def test_evaluate_default_mode_invariance(world, monkeypatch):
    """User batching changes nothing, bit for bit; a permuted pool keeps the rank of every target whose score is unique in
    the user's row; ranks agree with top_k's lists."""
    base = run_evaluate(world)
    assert base.fallback_units == 0
    monkeypatch.setattr(recommend, "PAIR_BUDGET", world["pool"][0].size * 7)      # batches of 7 users
    split = run_evaluate(world)
    for a, b in zip(host(base), host(split)):
        assert np.array_equal(a, b, equal_nan=True)
    monkeypatch.undo()
    pn, pf, pl = world["pool"]
    perm = np.random.default_rng(9).permutation(pn.size)
    shuffled = dict(world, exclude=world["exclude"][perm])
    sh = run_evaluate(shuffled, pool=(pn[perm], pf[perm], pl[perm]))
    imp = world["imp"]
    with torch.no_grad():
        plan = recommend.plan(world["model"], world["cache"], pn, pf, pl, exclude=world["exclude"])
        top = recommend.top_k(world["model"], world["cache"], plan, imp.hist_news, imp.hist_mask, imp.hist_fresh, imp.hist_life,
                              pn.size)
    news, score, count = top.news.cpu().numpy(), top.score.cpu().numpy(), top.count.cpu().numpy()
    rank, rank_sh = base.rank.cpu().numpy(), sh.rank.cpu().numpy()
    assert np.array_equal(base.eligible.cpu().numpy(), count)
    tn = world["targets"][0]
    checked = 0
    for u in range(rank.shape[0]):
        for t in range(rank.shape[1]):
            r = rank[u, t]
            assert (r > 0) == (rank_sh[u, t] > 0)
            if r > 0:
                assert news[u, r - 1] == tn[u, t]
                if np.sum(score[u, :count[u]] == score[u, r - 1]) == 1:
                    assert rank_sh[u, t] == r
                    checked += 1
    assert checked > 100


def test_evaluate_rejects_bad_arguments(world):
    imp, (tn, tm) = world["imp"], world["targets"]
    with torch.no_grad():
        plan = recommend.plan(world["model"], world["cache"], *world["pool"])
    ev = lambda tn, tm, **kw: recommend.evaluate(world["model"], world["cache"], plan, imp.hist_news, imp.hist_mask,
                                                 imp.hist_fresh, imp.hist_life, tn, tm, **kw)
    bad = tn.copy()
    bad[0, 0] = world["news"].news_num
    with pytest.raises(ValueError, match="target news ids"):
        ev(bad, tm)
    bad[0, 0] = -1
    with pytest.raises(ValueError, match="target news ids"):
        ev(bad, tm)
    wide = np.ones((tn.shape[0], 257), np.int64)
    with pytest.raises(ValueError, match="targets per user"):
        ev(wide, wide > 0)
    for cutoffs in ((0,), tuple(range(1, 10)), (2.5,)):
        with pytest.raises(ValueError, match="cutoffs"):
            ev(tn, tm, cutoffs=cutoffs)
