"""Host logic of the pool recommender (no GPU): the pool plan, the per-user unit replication and the pool checks."""
import numpy as np
import pytest
import torch

from lime_cikm25_b200 import engine, recommend


def _pool(n, seed, nb=10):
    rng = np.random.default_rng(seed)
    fresh = np.exp(rng.uniform(0, np.log(1e7), n)).astype(np.float32)
    life = np.exp(rng.uniform(np.log(600), np.log(6e5), n)).astype(np.float32)
    bp = torch.from_numpy(engine._host_bucket_pairs(fresh, life, nb))
    topic = torch.from_numpy(rng.integers(0, 40, n))
    return bp, topic


@pytest.mark.parametrize("n,limit", [(1, 38), (37, 38), (5000, 38), (5000, 7), (300, 1)])
def test_plan_pool_units(n, limit):
    bp, topic = _pool(n, n + limit)
    order, p0, cnt = engine.plan_pool(bp, topic, limit)
    assert torch.equal(torch.sort(order).values, torch.arange(n))                  # a permutation
    sbp, stp = bp[order], topic[order]
    key = sbp * 1000 + stp
    assert bool((key[1:] >= key[:-1]).all())                                         # sorted by (bucket pair, topic)
    assert int(cnt.sum()) == n and bool((cnt >= 1).all()) and bool((cnt <= limit).all())
    assert torch.equal(p0[1:], (p0 + cnt)[:-1]) and int(p0[0]) == 0                  # every position in exactly one unit
    for a, c in zip(p0.tolist(), cnt.tolist()):
        assert int(sbp[a:a + c].unique().numel()) == 1                               # never straddles a bucket-pair group
    # greedy cut: only the last unit of a group may hold fewer than limit candidates
    groups = torch.unique_consecutive(sbp, return_counts=True)[1]
    assert p0.numel() == int(((groups + limit - 1) // limit).sum())


def test_plan_pool_is_stable():
    bp = torch.tensor([4, 2, 4, 2, 4, 2, 4])
    topic = torch.tensor([1, 0, 1, 0, 0, 0, 1])
    order, _, _ = engine.plan_pool(bp, topic, 38)
    assert order.tolist() == [1, 3, 5, 4, 0, 2, 6]


def test_plan_pool_on_empty_pool():
    order, p0, cnt = engine.plan_pool(torch.zeros(0, dtype=torch.long), torch.zeros(0, dtype=torch.long), 38)
    assert order.numel() == p0.numel() == cnt.numel() == 0


class _Plan:
    """A PoolPlan stand-in on the CPU with a fixed unit template."""

    def __init__(self, C, p0, cnt):
        self.size, self.news = C, torch.arange(1, C + 1, dtype=torch.int32)
        self.fresh, self.life = torch.rand(C), torch.rand(C)
        self.remaining = torch.rand(C)
        self._t = (torch.tensor(p0, dtype=torch.int32), torch.tensor(cnt, dtype=torch.int32))
        self.limits = []

    def units(self, limit):
        self.limits.append(limit)
        return self._t


def test_from_pool_replicates_the_unit_template(monkeypatch):
    monkeypatch.setattr(engine, "choose_tile_c", lambda H: 39 if H <= 56 else 16)
    monkeypatch.setattr(engine._lib, "load", lambda: type("L", (), {"lime_score_scratch_ints": staticmethod(lambda n: 4 + n)})())
    C, Ub, H = 7, 3, 5
    plan = _Plan(C, [0, 2, 3], [2, 1, 4])
    hm = torch.ones(Ub, H, dtype=torch.bool)
    d = engine.DeviceImpressions.from_pool(plan, torch.ones(Ub, H, dtype=torch.int32), hm, torch.ones(Ub, H), torch.ones(Ub, H))
    assert plan.limits == [38]
    assert (d.num_units, d.num_pairs, d.num_impressions, d.max_history) == (9, Ub * C, Ub, H)
    assert d.dev["unit_imp"].tolist() == [0, 0, 0, 1, 1, 1, 2, 2, 2]
    assert d.dev["unit_pair0"].tolist() == [0, 2, 3, 7, 9, 10, 14, 16, 17]
    assert d.dev["unit_count"].tolist() == [2, 1, 4] * 3
    assert torch.equal(d.dev["cand_news"], plan.news.repeat(Ub))
    assert torch.equal(d.dev["cand_remaining"], plan.remaining.repeat(Ub))
    assert d.work_counter.numel() == 4 + 9 and d.planned_buckets is None
    d = engine.DeviceImpressions.from_pool(plan, torch.ones(Ub, 200, dtype=torch.int32), torch.ones(Ub, 200, dtype=torch.bool),
                                           torch.ones(Ub, 200), torch.ones(Ub, 200))
    assert plan.limits[-1] == 16                                     # long histories: the exact kernel's tile


def test_pool_validation():
    ok = dict(pool_fresh=[1.0, 2.0, 3.0], pool_life=[10.0, 20.0, 30.0])
    news, fresh, life, exc = recommend.validate_pool(10, [3, 1, 9], **ok)
    assert news.dtype == np.int32 and news.tolist() == [3, 1, 9] and exc is None
    with pytest.raises(ValueError, match="ids"):
        recommend.validate_pool(10, [3, 0, 9], **ok)                 # id 0 is the padding news
    with pytest.raises(ValueError, match="ids"):
        recommend.validate_pool(10, [3, 1, 10], **ok)                # out of range
    with pytest.raises(ValueError, match="ids"):
        recommend.validate_pool(10, [3, -1, 4], **ok)
    with pytest.raises(ValueError, match="same length"):
        recommend.validate_pool(10, [3, 1], **ok)
    with pytest.raises(ValueError, match="same length"):
        recommend.validate_pool(10, [3, 1, 4], pool_fresh=[1.0, 2.0, 3.0], pool_life=[1.0])
    with pytest.raises(ValueError, match="exclude"):
        recommend.validate_pool(10, [3, 1, 4], exclude=[0, 1], **ok)
    with pytest.raises(ValueError, match="at most once"):
        recommend.validate_pool(10, [3, 1, 3], **ok)
    with pytest.raises(ValueError, match="finite"):
        recommend.validate_pool(10, [3, 1, 4], pool_fresh=[1.0, np.nan, 3.0], pool_life=[1.0, 2.0, 3.0])
    with pytest.raises(ValueError, match="non-empty"):
        recommend.validate_pool(10, [], pool_fresh=[], pool_life=[])


def test_remaining_lifetime_rules():
    from types import SimpleNamespace
    from lime_cikm25_b200.util import remaining_lifetime
    fresh = np.asarray([10.0, 20.0], np.float32)
    cats = lambda: np.asarray([2, 0])
    assert remaining_lifetime(SimpleNamespace(lifetime_type="user_topic"), fresh, cats) is None
    r = remaining_lifetime(SimpleNamespace(lifetime_type="fixed", fixed_lifetime=100), fresh, cats)
    assert r.dtype == np.float32 and r.tolist() == [90.0, 80.0]
    r = remaining_lifetime(SimpleNamespace(lifetime_type="topic_wise", category_lifetime_map=torch.tensor([50.0, 0.0, 70.0])), fresh, cats)
    assert r.dtype == np.float32 and r.tolist() == [60.0, 30.0]
    with pytest.raises(ValueError):
        remaining_lifetime(SimpleNamespace(lifetime_type="other"), fresh, cats)
