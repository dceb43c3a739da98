"""Host-side checks of extend_news_cache / refresh_news_cache inputs (no GPU): everything that could index outside the
model's tables or the cache is rejected before a launch."""
import dataclasses

import numpy as np
import pytest
import torch

from lime_cikm25_b200 import synth, util


@pytest.fixture
def news():
    t = synth.make_news_table(20, vocabulary_size=300, seed=2)
    return dataclasses.replace(t, **{f: getattr(t, f)[1:] for f in
                                     ("title_text", "title_mask", "body_text", "body_mask", "category", "subCategory")})


def test_validate_news_accepts_and_casts(news):
    title, body, cat, sub = util.validate_news(news, 300, 18, 270)
    assert title.shape == (20, 32) and body.shape == (20, 128) and cat.shape == sub.shape == (20,)
    assert all(a.dtype == np.int32 and a.flags.c_contiguous for a in (title, body, cat, sub))
    assert np.array_equal(title, news.title_text) and np.array_equal(sub, news.subCategory)
    empty = dataclasses.replace(news, title_text=news.title_text[:0], body_text=news.body_text[:0],
                                category=news.category[:0], subCategory=news.subCategory[:0])
    assert util.validate_news(empty, 300, 18, 270)[0].shape == (0, 32)


@pytest.mark.parametrize("change", [
    dict(title_text=lambda a: a[:, :31]), dict(body_text=lambda a: a[:, :127]), dict(title_text=lambda a: a[:, :, None]),
    dict(title_text=lambda a: np.where(a > 0, 300, 0)), dict(body_text=lambda a: a - 1),
    dict(title_text=lambda a: a.astype(np.float32)), dict(body_text=lambda a: a[:19]),
    dict(category=lambda a: a + 18), dict(category=lambda a: a - 1 - a.max()), dict(subCategory=lambda a: a + 270),
    dict(subCategory=lambda a: a[:19]), dict(category=lambda a: a.reshape(20, 1)),
    dict(title_text=lambda a: np.where(a > 0, 2 ** 32 + 1, 0)),           # would wrap to a valid int32 id
])
def test_validate_news_rejects(news, change):
    bad = dataclasses.replace(news, **{k: f(getattr(news, k)) for k, f in change.items()})
    with pytest.raises(ValueError):
        util.validate_news(bad, 300, 18, 270)


def test_validate_refresh_rows():
    assert util.validate_refresh_rows([3, 1, 9], 10, 3).tolist() == [3, 1, 9]
    assert util.validate_refresh_rows(torch.tensor([4, 2]), 10, 2).dtype == np.int64
    assert util.validate_refresh_rows(np.zeros(0, np.int64), 10, 0).size == 0
    for rows, n in (([0, 1], 2), ([1, 10], 2), ([-1, 2], 2), ([2, 2], 2), ([1, 2], 3), ([[1, 2]], 2), ([1.0, 2.0], 2)):
        with pytest.raises(ValueError):
            util.validate_refresh_rows(rows, 10, n)


def test_capacity_nbytes_counts_headroom():
    bufs = (torch.zeros(10, 852), torch.zeros(10, 1720), torch.zeros(10 + 3, 2400, dtype=torch.float16), torch.zeros(10, 8),
            torch.zeros(10, 800))
    cache = util.NewsVectorCache(None, None, buffers=bufs)
    cache._set_rows(4, 3)
    row = (852 + 1720 + 8 + 800) * 4 + 2400 * 2
    assert cache.news_num == 4 and cache.capacity == 10
    assert cache.nbytes() == 4 * row + 3 * 2400 * 2
    assert cache.capacity_nbytes() == 10 * row + 3 * 2400 * 2
