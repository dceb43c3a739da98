"""Top-k recommendation over a news pool on the GPU: lime_pool_topk against a NumPy reference (exact indices, scores and
counts), and recommend.plan / recommend.top_k against the materialised impression set (every user one impression whose
candidates are the pool in the caller's order)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import lime_cikm25_b200 as L  # noqa: E402
from lime_cikm25_b200 import engine, ops, recommend, synth, util  # noqa: E402
from oracle.ref_import import make_config  # noqa: E402

DEV = "cuda"


# ---- kernel ----------------------------------------------------------------------------------------------------------
def ref_topk(scores, k, pool_index, pool_news=None, exclude=None, hist_news=None, hist_mask=None):
    """lexsort on (-score, pool_index) after the exclusions; NaN never returned."""
    U, C = scores.shape
    idx = np.full((U, k), -1, np.int64)
    val = np.full((U, k), -np.inf, np.float32)
    cnt = np.zeros(U, np.int64)
    for u in range(U):
        ok = ~np.isnan(scores[u])
        if exclude is not None:
            ok &= exclude == 0
        if hist_news is not None:
            ok &= ~np.isin(pool_news, hist_news[u][hist_mask[u] != 0])
        pos = np.nonzero(ok)[0]
        o = pos[np.lexsort((pool_index[pos], -scores[u, pos]))][:k]
        cnt[u] = o.size
        idx[u, :o.size] = pool_index[o]
        val[u, :o.size] = scores[u, o]
    return idx, val, cnt


def make_scores(U, C, dist, rng):
    if dist == "random":
        return rng.standard_normal((U, C)).astype(np.float32)
    if dist == "ties":                                  # a few distinct values: the boundary falls inside a run of ties
        return (rng.integers(-2, 3, (U, C)) * 0.5).astype(np.float32)
    vals = np.asarray([-0.0, 0.0, np.nan, 1.5, -1.5, np.inf, -np.inf], np.float32)     # signed zeros, NaN, infinities
    return vals[rng.integers(0, vals.size, (U, C))]


def run_kernel(scores, k, pool_index, pool_news=None, exclude=None, hist_news=None, hist_mask=None):
    t = lambda a, dt: None if a is None else torch.as_tensor(a).to(DEV, dt).contiguous()
    i, v, c = ops.pool_topk(t(scores, torch.float32), k, t(pool_index, torch.int32), t(pool_news, torch.int32),
                            t(exclude, torch.uint8), t(hist_news, torch.int32), t(hist_mask, torch.uint8))
    return i.cpu().numpy(), v.cpu().numpy(), c.cpu().numpy()


def check(got, want):
    gi, gv, gc = got
    wi, wv, wc = want
    assert np.array_equal(gc, wc)
    assert np.array_equal(gi, wi)
    assert np.array_equal(gv, wv)           # -0.0 == +0.0; -inf padding equal


@pytest.mark.parametrize("U,C,k", [(1, 1, 1), (1, 37, 10), (3, 37, 1024), (5, 4097, 10), (300, 4097, 100),
                                   (2, 300000, 1024), (1, 300000, 10), (4, 65238, 100)])
@pytest.mark.parametrize("dist", ["random", "ties", "special"])
def test_pool_topk_matches_reference(lib, U, C, k, dist):
    rng = np.random.default_rng(U * 7 + C + k)
    scores = make_scores(U, C, dist, rng)
    pool_index = rng.permutation(C).astype(np.int32)
    check(run_kernel(scores, k, pool_index), ref_topk(scores, k, pool_index))


@pytest.mark.parametrize("U,C,k,H", [(3, 37, 10, 5), (4, 4097, 100, 200), (2, 300000, 1024, 200), (200, 5000, 1024, 50)])
def test_pool_topk_exclusions(lib, U, C, k, H):
    """exclude mask + clicked history (H up to 224): pool news in the masked-in history are dropped, padding slots
    (mask 0, id 0 or a pool news) drop nothing."""
    rng = np.random.default_rng(C + H)
    scores = make_scores(U, C, "ties", rng)
    pool_index = rng.permutation(C).astype(np.int32)
    pool_news = rng.permutation(np.arange(1, C + 1)).astype(np.int32)
    exclude = (rng.random(C) < 0.2).astype(np.uint8)
    hist_news = rng.integers(1, 2 * C, (U, H)).astype(np.int32)          # about half of the clicks are in the pool
    hist_mask = rng.random((U, H)) < 0.7
    hist_news[:, -3:] = np.where(hist_mask[:, -3:], 0, pool_news[:3])     # padding: id 0, or a pool news masked out
    hist_mask[:, -3:] = False
    want = ref_topk(scores, k, pool_index, pool_news, exclude, hist_news, hist_mask)
    check(run_kernel(scores, k, pool_index, pool_news, exclude, hist_news, hist_mask), want)


def test_pool_topk_edge_counts(lib):
    rng = np.random.default_rng(3)
    C = 50
    scores = rng.standard_normal((3, C)).astype(np.float32)
    pool_index = np.arange(C, dtype=np.int32)
    exclude = np.zeros(C, np.uint8)
    exclude[10:] = 1                                                     # 10 returnable < k
    check(run_kernel(scores, 32, pool_index, exclude=exclude), ref_topk(scores, 32, pool_index, exclude=exclude))
    i, v, c = run_kernel(scores, 5, pool_index, exclude=np.ones(C, np.uint8))     # everything excluded
    assert (c == 0).all() and (i == -1).all() and np.isneginf(v).all()
    nan = np.full((2, C), np.nan, np.float32)
    i, v, c = run_kernel(nan, 1, pool_index)
    assert (c == 0).all() and (i == -1).all()


def test_pool_topk_rejects_bad_arguments(lib):
    s = torch.zeros(2, 8, device=DEV)
    pi = torch.arange(8, dtype=torch.int32, device=DEV)
    for k in (0, 1025):
        with pytest.raises(L._lib.LimeError, match="k="):
            ops.pool_topk(s, k, pi)
    o = torch.empty(2, 4, dtype=torch.int32, device=DEV)
    rc = lib.lime_pool_topk(s.data_ptr(), 2, 8, None, None, None, None, None, 0, 4, o.data_ptr(), o.data_ptr(), o.data_ptr(),
                            None, None)
    assert rc != 0 and b"null" in lib.lime_last_error()
    rc = lib.lime_pool_topk(s.data_ptr(), 2, 1 << 31, pi.data_ptr(), None, None, None, None, 0, 4, o.data_ptr(), o.data_ptr(),
                            o.data_ptr(), None, None)
    assert rc != 0 and b"pool" in lib.lime_last_error()


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
    pool_fresh = np.exp(rng.uniform(np.log(60.0), np.log(3e5), C)).astype(np.float32)       # freshness at request time
    pool_life = np.exp(rng.uniform(np.log(3600.0), np.log(6e5), C)).astype(np.float32)
    imp = synth.make_impressions(40, news.news_num, cand_fixed=2, seed=6)
    imp.hist_news[1, :5] = pool_news[:5]                                   # clicked pool news
    imp.hist_mask[1, :5] = True
    imp.hist_mask[2] = False                                               # an empty history
    return dict(cfg=cfg, model=model, news=news, cache=cache, pool=(pool_news, pool_fresh, pool_life), imp=imp)


def materialised(world, pool, remaining=None, users=None):
    """Every user one impression whose candidates are the pool in the caller's order -> scores [U, C] (the reference's
    full mini-batch prefix), the set and its DeviceImpressions."""
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
    return s.view(U, C).clone(), d


def run_top_k(world, k, pool=None, exclude=None, **kw):
    imp = world["imp"]
    with torch.no_grad():
        plan = recommend.plan(world["model"], world["cache"], *(pool or world["pool"]), exclude=exclude)
        return recommend.top_k(world["model"], world["cache"], plan, imp.hist_news, imp.hist_mask, imp.hist_fresh, imp.hist_life,
                               k, **kw)


def clicked(imp, u, news_ids):
    return np.isin(news_ids, imp.hist_news[u][imp.hist_mask[u]])


@pytest.fixture
def exact_mode():
    ops.score_configure(ops.SCORE_EXACT)
    yield
    ops.score_configure(ops.SCORE_AUTO)


@pytest.mark.parametrize("k", [1, 10, 100])
def test_top_k_exact_mode_matches_materialised_ranking(world, exact_mode, k):
    """(a) scores bit for bit equal to the materialised set's, indices = lime_rank_metrics' first k once clicked news
    are removed."""
    imp, pn = world["imp"], world["pool"][0]
    s, d = materialised(world, world["pool"])
    ranks, _ = ops.rank_metrics(s.reshape(-1), d.dev["labels"], d.dev["cand_off"])
    ranks = ranks.view(s.shape).cpu().numpy()
    res = run_top_k(world, k)
    idx, sc, cnt = res.index.cpu().numpy(), res.score.cpu().numpy(), res.count.cpu().numpy()
    s = s.cpu().numpy()
    for u in range(imp.num_impressions):
        order = np.argsort(ranks[u], kind="stable")
        order = order[~clicked(imp, u, pn[order])][:k]
        want = s[u, order]
        assert cnt[u] == order.size, (u, cnt[u], order.size)
        assert np.array_equal(idx[u, :cnt[u]], order), (u, idx[u, :cnt[u]], order, sc[u, :cnt[u]], want)
        nz = want != 0                                           # bit for bit; a -0.0 score is returned as +0.0
        assert np.array_equal(sc[u, :cnt[u]], want) and np.array_equal(sc[u, :cnt[u]][nz].view(np.uint32), want[nz].view(np.uint32)), u
        assert np.array_equal(res.news[u, :cnt[u]].cpu().numpy(), pn[order])
    assert clicked(imp, 1, pn[:5]).all() and not np.isin(pn[:5], res.news[1].cpu().numpy()).any()


def test_top_k_default_mode_within_tolerance(world):
    """(b) the tensor-core path: scores within 1e-5 of the exact kernel, no fallback units, top-k sets that differ only
    near the k-th score."""
    k = 20
    ops.score_configure(ops.SCORE_EXACT)
    try:
        s_exact, _ = materialised(world, world["pool"])
        want = run_top_k(world, k)
    finally:
        ops.score_configure(ops.SCORE_AUTO)
    res = run_top_k(world, k)
    assert res.fallback_units == 0
    s_exact = s_exact.cpu().numpy()
    floor = 0.1 * float(np.sqrt(np.mean(s_exact.astype(np.float64) ** 2)))
    idx, sc = res.index.cpu().numpy(), res.score.cpu().numpy()
    for u in range(idx.shape[0]):
        n = int(res.count[u])
        e = s_exact[u, idx[u, :n]]
        assert np.all(np.abs(sc[u, :n] - e) <= 1e-5 * np.maximum(np.abs(e), floor)), u
        kth = float(want.score[u, n - 1])
        diff = set(idx[u, :n]) ^ set(want.index[u, :n].cpu().numpy())
        for j in diff:
            assert abs(s_exact[u, j] - kth) <= 2e-5 * max(abs(kth), floor), (u, j)


def test_top_k_invariance(world, monkeypatch):
    """(c) user batching and pool order change nothing, bit for bit."""
    k = 15
    base = run_top_k(world, k)
    monkeypatch.setattr(recommend, "PAIR_BUDGET", world["pool"][0].size * 7)      # batches of 7 users
    split = run_top_k(world, k)
    for a in ("index", "news", "score", "count"):
        assert torch.equal(getattr(base, a), getattr(split, a)), a
    pn, pf, pl = world["pool"]
    perm = np.random.default_rng(9).permutation(pn.size)
    shuffled = run_top_k(world, k, pool=(pn[perm], pf[perm], pl[perm]))
    assert torch.equal(shuffled.score, base.score) and torch.equal(shuffled.count, base.count)
    sc = base.score.cpu().numpy()
    for u in range(sc.shape[0]):                                                 # modulo the order inside exact ties
        n = int(base.count[u])
        uniq = np.asarray([np.sum(sc[u, :n] == x) == 1 for x in sc[u, :n]])
        assert np.array_equal(shuffled.news[u, :n].cpu().numpy()[uniq], base.news[u, :n].cpu().numpy()[uniq])
        assert np.array_equal(perm[shuffled.index[u, :n].cpu().numpy()][uniq], base.index[u, :n].cpu().numpy()[uniq])


def test_top_k_exclusions(world):
    """(d) exclude_clicked, the plan's exclude mask, and an empty history."""
    imp, (pn, _, _) = world["imp"], world["pool"]
    exclude = (np.random.default_rng(4).random(pn.size) < 0.3).astype(np.uint8)
    k = 600
    res = run_top_k(world, k, exclude=exclude)
    idx, news = res.index.cpu().numpy(), res.news.cpu().numpy()
    for u in range(imp.num_impressions):
        n = int(res.count[u])
        assert not clicked(imp, u, news[u, :n]).any()
        assert not exclude[idx[u, :n]].any()
        assert n == min(k, int(((exclude == 0) & ~clicked(imp, u, pn)).sum()))
        assert (idx[u, n:] == -1).all() and (news[u, n:] == -1).all()
    assert int(res.count[2]) == min(k, int((exclude == 0).sum()))              # empty history: nothing clicked
    kept = run_top_k(world, k, exclude=exclude, exclude_clicked=False)
    assert np.isin(pn[:5], kept.news[1].cpu().numpy()).sum() == (exclude[:5] == 0).sum()


@pytest.mark.parametrize("lifetime", ["fixed", "topic_wise"])
def test_top_k_lifetime_types(world, exact_mode, lifetime):
    """(e) the remaining lifetime of lifetime_type 'fixed' / 'topic_wise' (util.py:98-102)."""
    cfg, news = world["model"].config, world["news"]
    pn, pf, _ = world["pool"]
    saved = cfg.lifetime_type, cfg.category_lifetime_map
    cfg.lifetime_type = lifetime
    cfg.category_lifetime_map = torch.linspace(3600.0, 2e5, news.category_num)
    try:
        remaining = util.remaining_lifetime(cfg, pf, lambda: news.category[pn])
        s, _ = materialised(world, world["pool"], remaining=remaining)
        res = run_top_k(world, 50, exclude_clicked=False)
    finally:
        cfg.lifetime_type, cfg.category_lifetime_map = saved
    s = s.cpu().numpy()
    idx = res.index.cpu().numpy()
    got = np.take_along_axis(s, idx, 1)
    assert np.array_equal(res.score.cpu().numpy(), got)
    assert np.array_equal(-np.sort(-s, axis=1)[:, :50], got)


def test_top_k_long_history(world, exact_mode):
    """H > 56 (up to 224): the exact kernel with its own tile, the same scores as the materialised set."""
    imp = world["imp"]
    H = 100
    long = synth.make_impressions(6, world["news"].news_num, max_history=H, cand_fixed=2, seed=8)
    w = dict(world, imp=long)
    s, _ = materialised(w, world["pool"])
    res = run_top_k(w, 10, exclude_clicked=False)
    assert np.array_equal(res.score.cpu().numpy(), -np.sort(-s.cpu().numpy(), axis=1)[:, :10])
    assert imp.hist_news.shape[1] == 50
