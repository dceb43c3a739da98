"""Explaining a recommendation without a GPU: explain_reference.explain_from_vectors against score_from_vectors /
crown_user in fp64, Explanation.top_history on hand-built arrays, and recommend.explain's input checks."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import lime_cikm25_b200 as L
from lime_cikm25_b200 import engine, recommend, synth, util
from explain_reference import explain_from_vectors
from oracle import lime_oracle as O
from oracle.ref_import import make_config

H = 12
UN = 16          # batch_size: user-node rows


@pytest.fixture(scope="module")
def world():
    cfg = make_config(vocabulary_size=400, batch_size=UN, max_history_num=H, word_embedding_init="skip")
    model = L.Model(cfg)
    model.initialize()
    synth.synthetic_parameters(model, 5)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    rng = np.random.default_rng(3)
    ncat = sd[O.NEWS + "category_embedding.weight"].shape[0]
    nsub = sd[O.NEWS + "subCategory_embedding.weight"].shape[0]
    N = 7
    data = dict(hist_vec=torch.as_tensor(rng.standard_normal((H, 400)) * 0.3), hist_cat=rng.integers(0, ncat, H),
                hist_sub=rng.integers(0, nsub, H), cand_vec=torch.as_tensor(rng.standard_normal((N, 400)) * 0.3),
                cand_cat=rng.integers(0, ncat, N), cand_sub=rng.integers(0, nsub, N),
                fresh=np.exp(rng.uniform(np.log(60.0), np.log(3e5), N)).astype(np.float32),
                life=np.exp(rng.uniform(np.log(3600.0), np.log(6e5), N)).astype(np.float32))
    return cfg, sd, data


def _args(data, mask, remaining, prefix):
    d = data
    return (d["hist_vec"], d["hist_cat"], d["hist_sub"], mask, d["cand_vec"], d["cand_cat"], d["cand_sub"], remaining, prefix)


def _remaining(cfg, data, lifetime):
    saved = cfg.lifetime_type, cfg.category_lifetime_map
    cfg.lifetime_type = lifetime
    cfg.category_lifetime_map = torch.linspace(3600.0, 2e5, 300)
    try:
        r = util.remaining_lifetime(cfg, data["fresh"], lambda: data["cand_cat"])
    finally:
        cfg.lifetime_type, cfg.category_lifetime_map = saved
    return data["life"] - data["fresh"] if r is None else r


def _softmaxes(monkeypatch):
    """Record every torch.softmax output (crown_user's last two: the candidate-aware weights, then the pooling alpha)."""
    seen, real = [], torch.softmax
    monkeypatch.setattr(torch, "softmax", lambda *a, **kw: seen.append(real(*a, **kw)) or seen[-1])
    return seen


MASKS = {"none_masked": np.ones(H, bool), "some_masked": np.arange(H) % 3 != 1, "all_but_one": np.arange(H) == 4}


@pytest.mark.parametrize("prefix", [1, H // 2, H, H + 1, H + 5, H + UN, "per_candidate"])
@pytest.mark.parametrize("mask", sorted(MASKS))
@pytest.mark.parametrize("lifetime", ["fixed", "topic_wise", "user_topic"])
def test_decomposition_reconstructs_the_score(world, monkeypatch, prefix, mask, lifetime):
    """fp64: bias + sum_h contrib = score_from_vectors, and alpha / topic_attention are crown_user's softmaxes (1e-12),
    at prefixes below, at and above H (user-node rows in the GraphSAGE mean) up to H + user_nodes."""
    cfg, sd, data = world
    N = data["cand_vec"].shape[0]
    pre = np.asarray([1, H, H + 3, H + UN, 2, H - 1, H + 1])[:N] if prefix == "per_candidate" else prefix
    remaining = _remaining(cfg, data, lifetime)
    args = _args(data, MASKS[mask], remaining, pre)
    ex = explain_from_vectors(sd, cfg, *args, dtype=torch.float64)
    want = O.score_from_vectors(sd, cfg, *args, dtype=torch.float64)
    scale = float(want.abs().max())
    assert float((ex["bias"] + ex["contrib"].sum(dim=1) - want).abs().max()) <= 1e-12 * scale
    assert float((ex["score"] - want).abs().max()) <= 1e-12 * scale
    assert torch.equal(ex["weight"], O.lifetime_weight(torch.as_tensor(remaining).double(), cfg))
    d = data
    for n in range(N):                                    # one crown_user call per candidate: its two last softmaxes
        seen = _softmaxes(monkeypatch)
        O.score_from_vectors(sd, cfg, d["hist_vec"], d["hist_cat"], d["hist_sub"], MASKS[mask], d["cand_vec"][n:n + 1],
                             d["cand_cat"][n:n + 1], d["cand_sub"][n:n + 1], remaining[n:n + 1],
                             int(np.broadcast_to(pre, (N,))[n]), dtype=torch.float64)
        monkeypatch.undo()
        assert float((ex["alpha"][n] - seen[-1].reshape(H)).abs().max()) <= 1e-12
        assert float((ex["topic_attention"][n] - seen[-2].reshape(H)).abs().max()) <= 1e-12
    assert torch.allclose(ex["alpha"].sum(dim=1), torch.ones(N, dtype=torch.float64), rtol=0, atol=1e-12)


def test_float32_oracle(world):
    cfg, sd, data = world
    r = data["life"] - data["fresh"]
    ex = explain_from_vectors(sd, cfg, *_args(data, MASKS["some_masked"], r, H + 2))
    want = explain_from_vectors(sd, cfg, *_args(data, MASKS["some_masked"], r, H + 2), dtype=torch.float64)
    assert all(v.dtype == torch.float32 for v in ex.values())
    assert float((ex["score"].double() - want["score"]).abs().max()) <= 1e-5 * float(want["score"].abs().max())


# ---- Explanation.top_history ------------------------------------------------------------------------------------------
def _explanation(contrib, hist_mask, score=None):
    contrib = torch.as_tensor(contrib, dtype=torch.float32)
    U, k, Hh = contrib.shape
    score = torch.zeros(U, k) if score is None else torch.as_tensor(score, dtype=torch.float32)
    z = torch.zeros(U, k, Hh)
    return recommend.Explanation(score, torch.ones(U, k), torch.zeros(U, k), contrib, z, z, torch.as_tensor(hist_mask))


def test_top_history_order_ties_and_padding():
    contrib = [[[0.5, -1.0, 2.0, 0.5, 3.0], [1.0, 1.0, 1.0, 1.0, 1.0]],
               [[0.1, 0.2, 0.3, 0.4, 0.5], [-3.0, -2.0, -1.0, 0.0, -0.0]]]
    mask = np.asarray([[1, 1, 1, 1, 0], [0, 1, 0, 1, 0]], np.uint8)
    ex = _explanation(contrib, mask, score=[[1.0, 1.0], [1.0, float("nan")]])
    top = ex.top_history(3)
    assert top.dtype == torch.int64 and tuple(top.shape) == (2, 2, 3)
    assert top[0, 0].tolist() == [2, 0, 3]           # slot 4 (largest) is masked out; 0.5 tie by ascending slot
    assert top[0, 1].tolist() == [0, 1, 2]           # all equal: ascending slots
    assert top[1, 0].tolist() == [3, 1, -1]          # two masked-in slots: -1 pad
    assert top[1, 1].tolist() == [-1, -1, -1]        # padded pair (NaN score)
    top = ex.top_history(7)                          # m > H: padded with -1
    assert tuple(top.shape) == (2, 2, 7) and top[0, 0].tolist() == [2, 0, 3, 1, -1, -1, -1]
    assert ex.top_history(1)[:, :, 0].tolist() == [[2, 0], [3, -1]]
    for m in (0, -1, 1.5):
        with pytest.raises(ValueError):
            ex.top_history(m)


def test_top_history_negative_contributions_rank_after_positive():
    ex = _explanation([[[-0.5, -0.1, 0.0, -2.0]]], np.ones((1, 4), np.uint8))
    assert ex.top_history(4)[0, 0].tolist() == [2, 1, 0, 3]


# ---- recommend.explain input checks (raise before the library is touched) ---------------------------------------------
@pytest.fixture
def cpu_plan():
    news = torch.tensor([5, 9, 3, 12], dtype=torch.int32)
    f = torch.ones(4)
    return engine.PoolPlan(news=news, fresh=f, life=f, remaining=None, index=torch.arange(4, dtype=torch.int32), exclude=None,
                           bucket_pair=torch.zeros(4, dtype=torch.int64), topic=torch.zeros(4, dtype=torch.int32),
                           caller_news=news.long())


def _hist(U, Hh):
    return np.zeros((U, Hh), np.int32), np.ones((U, Hh), bool), np.ones((U, Hh), np.float32), np.ones((U, Hh), np.float32)


@pytest.mark.parametrize("news,Hh,msg", [
    ([[5, 9], [3, 4]], 8, "pool"),                  # 4 is a cache row outside the pool
    ([[5, 9], [3, 20]], 8, "pool"),                 # out of range (news_num 20)
    ([[5, -2], [3, 9]], 8, "pool"),                 # negative other than -1
    ([[5, 9]], 8, "one row per history"),           # fewer rows than users
    ([5, 9], 8, "one row per history"),             # 1-D
    (np.zeros((2, 0), np.int64), 8, "one row per history"),
    ([[5, 9], [3, 12]], 225, "max_history"),
])
def test_explain_rejects_bad_inputs(cpu_plan, news, Hh, msg):
    cache = SimpleNamespace(news_num=20)
    with pytest.raises(ValueError, match=msg):
        recommend.explain(None, cache, cpu_plan, *_hist(2, Hh), news)


def test_explain_rejects_mismatched_histories(cpu_plan):
    hn, hm, hf, hl = _hist(2, 8)
    with pytest.raises(ValueError, match="share one"):
        recommend.explain(None, SimpleNamespace(news_num=20), cpu_plan, hn, hm[:, :7], hf, hl, [[5, 9], [3, 12]])
