"""Live cache updates: lime_cache_write_rows bit for bit against the derivation it replaces (split_f16_pairs / news_meta /
interleave_vg), extend_news_cache and refresh_news_cache against full builds in every encoder mode, scores and
recommendations over appended news, and the host-side rejections."""
import dataclasses

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import lime_cikm25_b200 as L  # noqa: E402
from lime_cikm25_b200 import _lib, engine, ops, recommend, synth, util  # noqa: E402
from oracle.ref_import import make_config  # noqa: E402

DEV = "cuda"
MODES = ("fp32", "bf16", "fp32x3")
TOPIC_COLS = (("hist_rows", engine.HIST_TOPIC_ID), ("cand_rows", engine.CAND_TOPIC_ID), ("meta", 0))


def bits(t):
    """Integer view of a tensor: bitwise comparison that also covers NaN and signed zeros."""
    return t.contiguous().view({torch.float32: torch.int32, torch.float16: torch.int16}[t.dtype])


def make_model(mode="fp32"):
    cfg = make_config(vocabulary_size=5000, batch_size=32, word_embedding_init="skip")
    model = L.Model(cfg)
    model.initialize()
    synth.synthetic_parameters(model, 7)
    model = model.to(DEV).eval()
    eng = model.news_encoder.engine
    eng.bf16, eng.x3 = mode == "bf16", mode == "fp32x3"
    return model


def pick(news, index):
    """The news ``index`` (a slice or an index array) of a table, as a table of their own."""
    return dataclasses.replace(news, **{f: getattr(news, f)[index] for f in
                                        ("title_text", "title_mask", "body_text", "body_mask", "category", "subCategory")})


def rows_of(news, lo, hi):
    return pick(news, slice(lo, hi))


@pytest.fixture(scope="module")
def news(lib):
    return synth.make_news_table(3000, vocabulary_size=5000, seed=11)


# ---- 1. the kernel against the old derivation --------------------------------------------------------------------------

def random_rows(n, seed):
    g = torch.Generator().manual_seed(seed)
    hist = (torch.randn(n, 852, generator=g) * torch.logspace(-4, 1, 852)).to(DEV)
    cand = (torch.randn(n, 1720, generator=g) * torch.logspace(-4, 1, 1720)).to(DEV)
    hist[:, engine.HIST_TOPIC_ID].view(torch.int32).copy_(torch.randint(0, 1000, (n,), generator=g).to(DEV))
    cand[:, engine.CAND_TOPIC_ID].view(torch.int32).copy_(torch.randint(0, 1000, (n,), generator=g).to(DEV))
    r = torch.arange(n, device=DEV)
    for col, val in ((3, -0.0), (4, 0.0), (5, 100.0), (6, -7e4), (7, 3e36), (8, float("inf"))):
        cand[r % 97 == col, col] = val           # signed zeros, beyond the fp16 range after scaling, scaling overflow
    cand[r % 89 == 1, 401] = float("nan")
    cand[r % 83 == 2, 799] = float("-inf")
    cand[:, engine.CAND_ABSMAX] = 12345.0          # stale value: the kernel stamps the row's max |w| there
    return hist, cand


def canary_cache(news_num, tail):
    f = lambda *s: torch.full(s, -7.25, device=DEV)
    return (f(news_num, 852), f(news_num, 1720), torch.full((news_num + tail, 2400), -3.5, dtype=torch.float16, device=DEV),
            f(news_num, 8), f(news_num, 800))


@pytest.mark.parametrize("n", [1, 7, 1000, 65238])
def test_write_rows_matches_old_derivation(lib, n):
    hist, cand = random_rows(n, n)
    news_num, tail = n + 301, 13
    dst = torch.randperm(news_num, generator=torch.Generator().manual_seed(n))[:n].to(DEV)
    out = canary_cache(news_num, tail)
    ops.cache_write_rows(hist, cand, dst, out[0], out[1], out[2], out[3], out[4])
    ref_cand = cand.clone()
    ref16 = ops.split_f16_pairs(ref_cand, 3, absmax=ref_cand[:, engine.CAND_ABSMAX])
    want = (hist, ref_cand, ref16, engine.ScoringEngine.news_meta(hist, ref_cand), engine.interleave_vg(hist))
    untouched = torch.ones(news_num + tail, dtype=torch.bool, device=DEV)
    untouched[dst] = False
    canary = canary_cache(news_num, tail)
    for got, w, c in zip(out, want, canary):
        assert torch.equal(bits(got[dst]), bits(w))
        k = untouched[:got.shape[0]]
        assert torch.equal(bits(got[k]), bits(c[k]))            # rows not written keep the canary, the cand16 tail too
    assert bool(torch.isinf(out[1][:, engine.CAND_ABSMAX][dst][(torch.arange(n, device=DEV) % 89) == 1]).all())


def test_write_rows_in_place_and_argument_errors(lib):
    n = 300
    hist, cand = random_rows(n, 3)
    H, C = hist.clone(), cand.clone()
    c16, meta, vg = torch.empty(n + 5, 2400, dtype=torch.float16, device=DEV), torch.empty(n, 8, device=DEV), torch.empty(n, 800, device=DEV)
    ops.cache_write_rows(H, C, torch.arange(n, device=DEV), H, C, c16, meta, vg)      # the form build_news_cache uses
    ref_cand = cand.clone()
    assert torch.equal(bits(c16[:n]), bits(ops.split_f16_pairs(ref_cand, 3, absmax=ref_cand[:, engine.CAND_ABSMAX])))
    assert torch.equal(bits(H), bits(hist)) and torch.equal(bits(C), bits(ref_cand))
    assert torch.equal(bits(meta), bits(engine.ScoringEngine.news_meta(hist, ref_cand)))
    assert torch.equal(bits(vg), bits(engine.interleave_vg(hist)))
    # destinations outside [0, news_num) are skipped on the device
    out = canary_cache(n, 0)
    bad = torch.tensor([-1, n, 1 << 40], device=DEV)
    ops.cache_write_rows(hist[:3], cand[:3], bad, *out)
    for got, c in zip(out, canary_cache(n, 0)):
        assert torch.equal(bits(got), bits(c))
    # argument errors: null pointers, n < 0, an empty cache, misalignment; shapes at the wrapper
    ok = torch.arange(n, device=DEV)
    p = [hist.data_ptr(), cand.data_ptr(), n, ok.data_ptr(), H.data_ptr(), C.data_ptr(), c16.data_ptr(), meta.data_ptr(),
         vg.data_ptr(), n, None]
    for i, v in ((0, None), (3, None), (6, None), (8, None), (2, -1), (9, 0), (4, H.data_ptr() + 4), (3, ok.data_ptr() + 4)):
        args = list(p)
        args[i] = v
        assert lib.lime_cache_write_rows(*args) != 0
        assert b"lime_cache_write_rows" in lib.lime_last_error()
    with pytest.raises(_lib.LimeError):
        ops.cache_write_rows(hist[:, :851], cand, torch.arange(n, device=DEV), H, C, c16, meta, vg)
    with pytest.raises(_lib.LimeError):
        ops.cache_write_rows(hist, cand, torch.arange(n, device=DEV), H, C, c16[:n - 1], meta, vg)
    with pytest.raises(_lib.LimeError):
        ops.cache_write_rows(hist, cand, torch.arange(n, device=DEV, dtype=torch.int32), H, C, c16, meta, vg)


# ---- 2. extend == full build ----------------------------------------------------------------------------------------------

def assert_same_cache(a, b):
    """Every array bitwise equal (cand16 with its tail); topic-id columns up to one bijection of ids."""
    ids = []
    for name in ("hist_rows", "cand_rows", "cand16", "meta", "hist_vg"):
        x, y = getattr(a, name), getattr(b, name)
        assert x.shape == y.shape, name
        x, y = bits(x), bits(y)
        col = dict(TOPIC_COLS).get(name)
        if col is not None:
            ids.append((x[:, col].clone(), y[:, col].clone()))
            x, y = x.clone(), y.clone()
            x[:, col] = 0
            y[:, col] = 0
        assert torch.equal(x, y), name
    for (x, y) in ids[1:]:
        assert torch.equal(x, ids[0][0]) and torch.equal(y, ids[0][1])
    pairs = set(zip(ids[0][0].tolist(), ids[0][1].tolist()))
    assert len(pairs) == len(set(p[0] for p in pairs)) == len(set(p[1] for p in pairs))      # one bijection


def extended_cache(model, news, n0, n1, capacity):
    """build over news[:n0], extend by news[n0:n1], then by news[n1:]."""
    with torch.no_grad():
        cache = util.build_news_cache(model, rows_of(news, 0, n0), capacity=capacity)
        keep = cache.buffers[0].data_ptr()
        r1 = util.extend_news_cache(model, cache, rows_of(news, n0, n1))
        assert cache.buffers[0].data_ptr() == keep and cache.capacity == capacity        # inside the headroom
        r2 = util.extend_news_cache(model, cache, rows_of(news, n1, news.news_num))
        assert cache.capacity >= news.news_num and cache.capacity > capacity               # grown
    assert torch.equal(r1.cpu(), torch.arange(n0, n1)) and torch.equal(r2.cpu(), torch.arange(n1, news.news_num))
    assert r1.dtype == torch.int64 and r1.device.type == "cuda"
    return cache


@pytest.mark.parametrize("mode", MODES)
def test_extend_equals_full_build(lib, news, mode):
    m_ext, m_full = make_model(mode), make_model(mode)      # two registries: compact topic ids may differ
    cache = extended_cache(m_ext, news, 2000, 2500, 2600)
    with torch.no_grad():
        full = util.build_news_cache(m_full, news)
    assert cache.news_num == full.news_num == news.news_num
    assert_same_cache(cache, full)
    # holders of the cache object see the new arrays; the old rows stay where they were
    assert cache.hist_rows.data_ptr() == cache.buffers[0].data_ptr()


# ---- 3. scores and recommendations over appended news ----------------------------------------------------------------

@pytest.fixture(scope="module")
def pair(news):
    m_ext, m_full = make_model(), make_model()
    ext = extended_cache(m_ext, news, 2000, 2500, 2600)
    with torch.no_grad():
        full = util.build_news_cache(m_full, news)
    return m_ext, ext, m_full, full


@pytest.mark.parametrize("mode", [ops.SCORE_AUTO, ops.SCORE_EXACT])
def test_scores_over_appended_news(pair, news, mode):
    m_ext, ext, m_full, full = pair
    imp = synth.make_impressions(600, news.news_num, seed=12)
    assert (imp.cand_news >= 2000).any() and (imp.hist_news >= 2500).any()
    try:
        ops.score_configure(mode)
        with torch.no_grad():
            a = util.score_impressions(m_ext, ext, engine.DeviceImpressions(imp, DEV), 32).clone()
            b = util.score_impressions(m_full, full, engine.DeviceImpressions(imp, DEV), 32).clone()
    finally:
        ops.score_configure(ops.SCORE_AUTO)
    assert torch.equal(bits(a), bits(b))


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    floor = 0.1 * float(np.sqrt(np.mean(b * b))) + 1e-30
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), floor)))


def test_recommend_over_appended_news(pair, news):
    m_ext, ext, m_full, full = pair
    rng = np.random.default_rng(3)
    C = 600
    pool = np.concatenate([rng.choice(np.arange(1, 2000), C - 200, replace=False), rng.choice(np.arange(2000, news.news_num), 200, replace=False)])
    fresh = np.exp(rng.uniform(np.log(60.0), np.log(3e5), C)).astype(np.float32)
    life = np.exp(rng.uniform(np.log(3600.0), np.log(6e5), C)).astype(np.float32)
    imp = synth.make_impressions(50, news.news_num, cand_fixed=2, seed=4)
    U, T = imp.num_impressions, 6
    tn = pool[rng.integers(0, C, (U, T))].astype(np.int64)
    tm = np.ones((U, T), bool)
    hist = (imp.hist_news, imp.hist_mask, imp.hist_fresh, imp.hist_life)

    def run(model, cache):
        with torch.no_grad():
            plan = recommend.plan(model, cache, pool, fresh, life)
            top = recommend.top_k(model, cache, plan, *hist, 20)
            ev = recommend.evaluate(model, cache, plan, *hist, tn, tm, cutoffs=(10, 50))
        return top, ev

    try:
        ops.score_configure(ops.SCORE_EXACT)
        (ta, ea), (tb, eb) = run(m_ext, ext), run(m_full, full)
        assert torch.equal(ta.index, tb.index) and torch.equal(bits(ta.score), bits(tb.score))
        assert torch.equal(ea.rank, eb.rank) and torch.equal(ea.metrics.isnan(), eb.metrics.isnan())
        assert torch.equal(torch.nan_to_num(ea.metrics), torch.nan_to_num(eb.metrics))
    finally:
        ops.score_configure(ops.SCORE_AUTO)
    # default mode: plan_pool sorts by compact topic id, so unit cuts (and interpolation nodes) may differ
    (ta, ea), (tb, eb) = run(m_ext, ext), run(m_full, full)
    sa, sb = ta.score.cpu().numpy(), tb.score.cpu().numpy()
    assert rel(sa, sb) < 1e-5
    assert (ta.index == tb.index).float().mean() > 0.95
    # a pool of appended news only
    new = np.arange(2500, news.news_num)
    with torch.no_grad():
        plan = recommend.plan(m_ext, ext, new, fresh[:new.size], life[:new.size])
        top = recommend.top_k(m_ext, ext, plan, *hist, 10, exclude_clicked=False)
    got = top.news.cpu().numpy()
    assert (top.count.cpu().numpy() == 10).all() and np.isin(got, new).all()


# ---- 4. refresh ---------------------------------------------------------------------------------------------------------

def test_refresh(lib, news):
    model, m_full = make_model(), make_model()
    with torch.no_grad():
        cache = util.build_news_cache(model, news)
    before = {k: getattr(cache, k).clone() for k in ("hist_rows", "cand_rows", "cand16", "meta", "hist_vg")}
    imp = synth.make_impressions(600, news.news_num, seed=13)
    with torch.no_grad():
        s0 = util.score_impressions(model, cache, engine.DeviceImpressions(imp, DEV), 32).clone()
    rows = np.array([5, 17, 999, 2000, 2999], np.int64)
    edited = dataclasses.replace(news, **{f: getattr(news, f).copy() for f in ("title_text", "body_text", "category", "subCategory")})
    rng = np.random.default_rng(8)
    edited.title_text[rows] = rng.integers(1, 5000, (rows.size, 32))
    edited.body_text[rows[:2]] = rng.integers(1, 5000, (2, 128))
    edited.category[rows[1]], edited.subCategory[rows[1]] = edited.category[rows[4]], edited.subCategory[rows[4]]
    seen = set(zip(news.category.tolist(), news.subCategory.tolist()))
    fresh_topic = next((c, s) for c in range(news.category_num) for s in range(news.subCategory_num) if (c, s) not in seen)
    edited.category[rows[2]], edited.subCategory[rows[2]] = fresh_topic            # a topic no news had
    with torch.no_grad():
        order = rows[::-1].copy()                               # any order of the rows
        util.refresh_news_cache(model, cache, torch.from_numpy(order), pick(edited, order))
        full = util.build_news_cache(m_full, edited)
    assert_same_cache(cache, full)
    others = np.setdiff1d(np.arange(news.news_num), rows)
    for k, v in before.items():
        got = getattr(cache, k)
        assert torch.equal(bits(got[others]), bits(v[others])), k
        assert not torch.equal(bits(got[rows]), bits(v[rows])), k
    # scores of impressions that touch no refreshed row are unchanged
    touched = np.isin(imp.hist_news, rows).any(axis=1) | np.array(
        [np.isin(imp.cand_news[imp.cand_off[i]:imp.cand_off[i + 1]], rows).any() for i in range(imp.num_impressions)])
    assert touched.any() and (~touched).sum() > 100
    with torch.no_grad():
        s1 = util.score_impressions(model, cache, engine.DeviceImpressions(imp, DEV), 32)
    keep = np.concatenate([np.arange(imp.cand_off[i], imp.cand_off[i + 1]) for i in np.nonzero(~touched)[0]])
    keep = torch.from_numpy(keep).to(DEV)
    assert torch.equal(bits(s1[keep]), bits(s0[keep]))


# ---- 5. rejections ------------------------------------------------------------------------------------------------------

def test_rejections(lib, news):
    model = make_model()
    with torch.no_grad():
        cache = util.build_news_cache(model, rows_of(news, 0, 100))
    add = rows_of(news, 100, 110)
    n0 = cache.news_num
    empty = util.extend_news_cache(model, cache, rows_of(news, 100, 100))                  # n = 0: a no-op
    assert empty.numel() == 0 and empty.dtype == torch.int64 and cache.news_num == n0
    util.refresh_news_cache(model, cache, [], rows_of(news, 100, 100))

    def bad(**kw):
        return dataclasses.replace(add, **kw)
    vocab = 5000
    cases = [bad(title_text=add.title_text[:, :31]), bad(body_text=add.body_text[:, :127]),
             bad(title_text=np.where(add.title_text > 0, vocab, 0)), bad(body_text=add.body_text - 1),
             bad(category=add.category + news.category_num), bad(subCategory=np.full_like(add.subCategory, -1)),
             bad(category=add.category[:9])]
    for c in cases:
        with pytest.raises(ValueError):
            util.extend_news_cache(model, cache, c)
    for rows in ([0] + list(range(1, 10)), list(range(1, 10)) + [n0], [1, 2, 3, 4, 5, 6, 7, 8, 9, 9], list(range(1, 10)),
                 [-1] + list(range(2, 11))):
        with pytest.raises(ValueError):
            util.refresh_news_cache(model, cache, rows, add)
    assert cache.news_num == n0
    with torch.no_grad():
        next(model.parameters()).mul_(1.0)                        # a weight update (in place)
    with pytest.raises(ValueError, match="weights changed"):
        util.extend_news_cache(model, cache, add)
    with pytest.raises(ValueError, match="weights changed"):
        util.refresh_news_cache(model, cache, list(range(1, 11)), add)
    assert cache.news_num == n0
