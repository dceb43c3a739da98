"""Explaining a recommendation on the GPU: lime_explain_pairs against the fp64 reference
(explain_reference.explain_from_vectors on the GPU-built LIME vectors) at every history length class and GraphSAGE prefix
class, the decomposition identities, agreement with top_k, invariance to how the lists are batched, padding, and rejection
of bad inputs before any launch."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import lime_cikm25_b200 as L  # noqa: E402
from lime_cikm25_b200 import engine, ops, recommend, synth  # noqa: E402
from explain_reference import explain_from_vectors  # noqa: E402
from oracle import lime_oracle as O  # noqa: E402
from oracle.ref_import import make_config  # noqa: E402

DEV = "cuda"
UN = 32                      # config.batch_size: user-node rows
K = 5                        # news explained per user in the parity cases
# Bars against fp64: about 3x the worst error measured on one B200 (1,000 W power limit) for these seeded inputs.
# score / weight: rel() of test_gpu_parity; bias / contrib: per pair, against |bias| + sum_h |contrib|; alpha / topic
# attention: absolute.
# Worst measured: score 1.5e-6, weight 1.7e-7, bias 4.1e-8, contrib 6.3e-7, alpha 1.2e-7, topic attention 2.3e-7.
BAR = {"score": 5e-6, "weight": 5e-7, "bias": 1.2e-7, "contrib": 2e-6, "alpha": 3.5e-7, "topic_attention": 7e-7}


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    floor = 0.1 * float(np.sqrt(np.mean(b * b))) + 1e-30
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), floor)))


@pytest.fixture(scope="module")
def world(lib):
    # sigmoid_scaling_alpha 3e-5 / s: lifetime weights spread over (0, 1) on these hour-scale lifetimes (at the default 0.3 / s
    # they are 0 or 1), so a contribution that misses w shows
    cfg = make_config(vocabulary_size=5000, batch_size=UN, word_embedding_init="skip", sigmoid_scaling_alpha=3e-5)
    model = L.Model(cfg)
    model.initialize()
    synth.synthetic_parameters(model, 7)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    model = model.to(DEV).eval()
    news = synth.make_news_table(3000, vocabulary_size=5000, seed=11)
    from lime_cikm25_b200 import util
    with torch.no_grad():
        cache = util.build_news_cache(model, news)
    rng = np.random.default_rng(5)
    C = 700
    pool_news = rng.choice(np.arange(1, news.news_num), C, replace=False).astype(np.int32)
    pool_fresh = np.exp(rng.uniform(np.log(60.0), np.log(3e5), C)).astype(np.float32)
    pool_life = np.exp(rng.uniform(np.log(3600.0), np.log(6e5), C)).astype(np.float32)
    return dict(cfg=cfg, model=model, sd=sd, news=news, cache=cache, pool=(pool_news, pool_fresh, pool_life))


def make_plan(world, lifetime="user_topic"):
    cfg = world["cfg"]
    saved = cfg.lifetime_type, cfg.category_lifetime_map
    cfg.lifetime_type = lifetime
    cfg.category_lifetime_map = torch.linspace(3600.0, 2e5, world["news"].category_num)
    try:
        with torch.no_grad():
            return recommend.plan(world["model"], world["cache"], *world["pool"])
    finally:
        cfg.lifetime_type, cfg.category_lifetime_map = saved


@pytest.fixture(scope="module")
def plan(world):
    return make_plan(world)


def histories(world, U, H, seed):
    """[U, H] histories: user 0 with no slot masked, user 1 with every slot masked but one, the rest random masks."""
    imp = synth.make_impressions(U, world["news"].news_num, max_history=H, cand_fixed=1, seed=seed)
    hm = imp.hist_mask.copy()
    hm[0] = True
    if U > 1:
        hm[1] = False
        hm[1, H // 3] = True
    return imp.hist_news.astype(np.int32), hm, imp.hist_fresh.astype(np.float32), imp.hist_life.astype(np.float32)


def pick_news(world, U, k, seed):
    rng = np.random.default_rng(seed)
    pn = world["pool"][0]
    return np.stack([rng.choice(pn, k, replace=False) for _ in range(U)]).astype(np.int64)


def kernel_explain(world, plan, news, hist, prefix):
    """lime_explain_pairs on DeviceImpressions.from_lists at a given GraphSAGE prefix -> dict of [U, k(, H)] numpy arrays
    (news without padding, so the pair order is the caller's)."""
    cache, model = world["cache"], world["model"]
    hn, hm, hf, hl = (torch.as_tensor(a).to(DEV) for a in hist)
    nw = torch.as_tensor(news).to(DEV, torch.int64)
    U, k = nw.shape
    d = engine.DeviceImpressions.from_lists(plan, cache.news_num, nw, hn, hm, hf, hl)
    assert torch.equal(d.order, torch.arange(k, device=DEV).expand(U, k))
    H = d.max_history
    vec = torch.full((3, U * k), float("nan"), device=DEV)
    mat = torch.full((3, U * k, H), float("nan"), device=DEV)
    with torch.no_grad():
        ops.explain_pairs(model.scoring.cache_struct(cache.hist_rows, cache.cand_rows), d.struct(), prefix, vec[0], mat[1], mat[2],
                          mat[0], vec[2], vec[1], d.work_counter)
    v, m = vec.view(3, U, k).cpu().numpy(), mat.view(3, U, k, H).cpu().numpy()
    return dict(score=v[0], weight=v[1], bias=v[2], contrib=m[0], alpha=m[1], topic_attention=m[2])


def oracle_explain(world, plan, news, hist, prefix):
    """explain_from_vectors in fp64 on the cache's LIME vectors, the plan's freshness / lifetime / remaining."""
    cache, se, nt, sd, cfg = world["cache"], world["model"].scoring, world["news"], world["sd"], world["cfg"]
    hn, hm, hf, hl = hist
    pos = plan.positions(cache.news_num).cpu().numpy()[news]
    fresh, life = plan.fresh.cpu().numpy()[pos], plan.life.cpu().numpy()[pos]
    remaining = plan.remaining.cpu().numpy()[pos] if plan.remaining is not None else life - fresh
    vec = lambda ids, f, l_: se.lime_vectors(cache.hist_rows[torch.as_tensor(ids).long().to(DEV)], torch.as_tensor(f).to(DEV),
                                             torch.as_tensor(l_).to(DEV)).cpu()
    out = []
    for u in range(news.shape[0]):
        hv, cv = vec(hn[u], hf[u], hl[u]), vec(news[u], fresh[u], life[u])
        out.append(explain_from_vectors(sd, cfg, hv, nt.category[hn[u]], nt.subCategory[hn[u]], hm[u], cv, nt.category[news[u]],
                                          nt.subCategory[news[u]], remaining[u], prefix, torch.float64))
    return {n: np.stack([o[n].numpy() for o in out]) for n in out[0]}


def errors(got, want):
    scale = np.maximum(np.abs(want["bias"]) + np.abs(want["contrib"]).sum(-1), 1e-30)    # [U, k]
    return dict(score=rel(got["score"], want["score"]), weight=rel(got["weight"], want["weight"]),
                bias=float(np.max(np.abs(got["bias"] - want["bias"]) / scale)),
                contrib=float(np.max(np.abs(got["contrib"] - want["contrib"]).max(-1) / scale)),
                alpha=float(np.max(np.abs(got["alpha"] - want["alpha"]))),
                topic_attention=float(np.max(np.abs(got["topic_attention"] - want["topic_attention"]))))


def check_parity(got, want, tag):
    err = errors(got, want)
    print("explain-err", tag, " ".join("%s=%.2e" % kv for kv in err.items()))
    for n, e in err.items():
        assert e <= BAR[n], (tag, n, e)


@pytest.mark.parametrize("H", [1, 8, 50, 56, 57, 112, 200, 224])
def test_fp64_parity_history_and_prefix(world, plan, H):
    """Every output against fp64 at prefixes 1, H/2, H, H + 1 and H + user_nodes (the user-node rows of the GraphSAGE
    mean), histories with no slot masked, all but one masked, and random masks."""
    hist = histories(world, 3, H, seed=H)
    news = pick_news(world, 3, K, seed=H)
    for prefix in sorted({1, max(1, H // 2), H, H + 1, H + UN}):
        got = kernel_explain(world, plan, news, hist, prefix)
        check_parity(got, oracle_explain(world, plan, news, hist, prefix), "H=%d P=%d" % (H, prefix))


@pytest.mark.parametrize("lifetime", ["fixed", "topic_wise", "user_topic"])
def test_fp64_parity_lifetime_types(world, lifetime):
    """The remaining lifetime of each lifetime_type (util.py:98-104) reaches the weight, the bias and every contribution."""
    p = make_plan(world, lifetime)
    assert (p.remaining is None) == (lifetime == "user_topic")
    hist = histories(world, 3, 50, seed=4)
    news = pick_news(world, 3, K, seed=4)
    got = kernel_explain(world, p, news, hist, UN)
    check_parity(got, oracle_explain(world, p, news, hist, UN), "lifetime=%s" % lifetime)


def run_top_k(world, plan, hist, k):
    with torch.no_grad():
        return recommend.top_k(world["model"], world["cache"], plan, *hist, k)


def run_explain(world, plan, hist, news):
    with torch.no_grad():
        return recommend.explain(world["model"], world["cache"], plan, *hist, news)


@pytest.fixture
def exact_mode():
    ops.score_configure(ops.SCORE_EXACT)
    yield
    ops.score_configure(ops.SCORE_AUTO)


@pytest.mark.parametrize("H", [50, 200])
def test_decomposition_of_top_k_lists(world, plan, H):
    """bias + sum_h contrib reconstructs the score to 1e-6 of |bias| + sum_h |contrib|; alpha and the candidate-aware
    weights each sum to 1 within 1e-6."""
    hist = histories(world, 40, H, seed=H + 1)
    res = run_top_k(world, plan, hist, 10)
    ex = run_explain(world, plan, hist, res.news)
    ok = (res.news >= 0).cpu().numpy()
    c = ex.contrib.double().cpu().numpy()[ok]
    b, s = ex.bias.double().cpu().numpy()[ok], ex.score.double().cpu().numpy()[ok]
    assert np.all(np.abs(b + c.sum(-1) - s) <= 1e-6 * (np.abs(b) + np.abs(c).sum(-1)))
    for a in (ex.alpha, ex.topic_attention):
        assert np.all(np.abs(a.double().cpu().numpy()[ok].sum(-1) - 1.0) <= 1e-6)
    w = ex.weight.cpu().numpy()[ok]
    assert np.all((w > 0) & (w < 1))


@pytest.mark.parametrize("H", [50, 200])
def test_exact_mode_scores_equal_top_k_bit_for_bit(world, plan, exact_mode, H):
    hist = histories(world, 40, H, seed=H + 2)
    res = run_top_k(world, plan, hist, 10)
    ex = run_explain(world, plan, hist, res.news)
    ok = res.news >= 0
    assert int(ok.sum()) > 0
    got, want = ex.score[ok].cpu().numpy(), res.score[ok].cpu().numpy()
    nz = want != 0                                               # top_k returns a -0.0 score as +0.0
    assert np.array_equal(got, want) and np.array_equal(got[nz].view(np.uint32), want[nz].view(np.uint32))


@pytest.mark.parametrize("H", [50, 200])
def test_default_mode_scores_agree_with_top_k(world, plan, H):
    """top_k's tensor-core scores (H <= 56) against the exact kernel explain runs: the suite's 5e-5 bar."""
    hist = histories(world, 40, H, seed=H + 3)
    res = run_top_k(world, plan, hist, 10)
    ex = run_explain(world, plan, hist, res.news)
    ok = (res.news >= 0).cpu().numpy()
    got, want = ex.score.cpu().numpy()[ok], res.score.cpu().numpy()[ok]
    floor = 0.1 * float(np.sqrt(np.mean(want.astype(np.float64) ** 2)))
    assert np.all(np.abs(got - want) <= 5e-5 * np.maximum(np.abs(want), floor))


def bits(ex):
    return [getattr(ex, n).contiguous().view(torch.int32) for n in ("score", "weight", "bias", "contrib", "alpha", "topic_attention")]


def test_invariance_to_batching(world, plan, monkeypatch):
    """The same [U, k] lists explained at once, column by column and in batches of 7 users give the same bits."""
    H = 50
    hist = histories(world, 40, H, seed=8)
    news = torch.as_tensor(pick_news(world, 40, 12, seed=8))
    whole = bits(run_explain(world, plan, hist, news))
    cols = [bits(run_explain(world, plan, hist, news[:, j:j + 1])) for j in range(news.shape[1])]
    for i, w in enumerate(whole):
        assert torch.equal(w, torch.cat([c[i] for c in cols], dim=1)), i
    monkeypatch.setattr(recommend, "EXPLAIN_BUDGET", 7 * 12 * (3 * H + 3))
    for w, s in zip(whole, bits(run_explain(world, plan, hist, news))):
        assert torch.equal(w, s)


def test_padding(world, plan):
    """-1 anywhere in a row (and a row of -1 only) gives NaN in every output and -1 in top_history; the other news get
    the bits they get without the padding."""
    H = 57
    hist = histories(world, 4, H, seed=9)
    news = pick_news(world, 4, 6, seed=9)
    padded = news.copy()
    padded[0, [1, 4]] = -1
    padded[1, 0] = -1
    padded[2] = -1
    ex = run_explain(world, plan, hist, padded)
    full = run_explain(world, plan, hist, news)
    pad = torch.as_tensor(padded < 0, device=DEV)
    for a, b in zip(bits(ex), bits(full)):
        a, b = a.view(4, 6, -1), b.view(4, 6, -1)
        assert torch.equal(a[~pad], b[~pad])
    for n in ("score", "weight", "bias", "contrib", "alpha", "topic_attention"):
        assert bool(torch.isnan(getattr(ex, n)[pad]).all()), n
    top = ex.top_history(5)
    assert bool((top[pad] == -1).all()) and bool((top[~pad][:, 0] >= 0).all())
    hm = torch.as_tensor(hist[1], device=DEV)
    t = top[~pad]
    owner = torch.arange(4, device=DEV).view(4, 1).expand(4, 6)[~pad]
    assert bool(hm[owner.view(-1, 1), t.clamp_min(0)][t >= 0].all())         # masked-in slots only


def test_rejects_bad_inputs_before_any_launch(world, plan, lib):
    cache, model = world["cache"], world["model"]
    hist = histories(world, 2, 8, seed=10)
    news = pick_news(world, 2, 3, seed=10)
    outside = np.setdiff1d(np.arange(1, cache.news_num), world["pool"][0])[0]
    bad = [news[:1], news[:, 0], np.where(np.arange(3) == 1, outside, news), np.where(np.arange(3) == 2, cache.news_num, news),
           np.where(np.arange(3) == 0, -2, news)]
    n0 = lib.lime_launch_count()
    for b in bad:
        with pytest.raises(ValueError):
            run_explain(world, plan, hist, b)
    long_hist = histories(world, 2, 225, seed=10)
    with pytest.raises(ValueError, match="max_history"):
        run_explain(world, plan, long_hist, news)
    assert lib.lime_launch_count() == n0
    # the C entry point: bad prefixes, H = 225 and a null output fail before any launch, the outputs keep their canary
    hn, hm, hf, hl = (torch.as_tensor(a).to(DEV) for a in hist)
    d = engine.DeviceImpressions.from_lists(plan, cache.news_num, torch.as_tensor(news).to(DEV), hn, hm, hf, hl)
    canary = -12345.678
    vec = torch.full((3, 6), canary, device=DEV)
    mat = torch.full((3, 6, 8), canary, device=DEV)
    cs = model.scoring.cache_struct(cache.hist_rows, cache.cand_rows)
    n0 = lib.lime_launch_count()
    for prefix in (0, 8 + UN + 1):
        with pytest.raises(L._lib.LimeError, match="prefix_main"):
            ops.explain_pairs(cs, d.struct(), prefix, vec[0], mat[1], mat[2], mat[0], vec[2], vec[1], d.work_counter)
    st = d.struct()
    st.max_history = 225
    rc = lib.lime_explain_pairs(cs, st, UN, vec[0].data_ptr(), mat[1].data_ptr(), mat[2].data_ptr(), mat[0].data_ptr(),
                                vec[2].data_ptr(), vec[1].data_ptr(), d.work_counter.data_ptr(), None)
    assert rc != 0 and b"max_history" in lib.lime_last_error()
    rc = lib.lime_explain_pairs(cs, d.struct(), UN, vec[0].data_ptr(), mat[1].data_ptr(), None, mat[0].data_ptr(),
                                vec[2].data_ptr(), vec[1].data_ptr(), d.work_counter.data_ptr(), None)
    assert rc != 0 and b"null" in lib.lime_last_error()
    torch.cuda.synchronize()
    assert lib.lime_launch_count() == n0
    assert bool((vec == canary).all()) and bool((mat == canary).all())
