"""lime_cikm25_b200 — B200-native (sm_100a) implementation of LIME's scoring hot path.

The sub-modules mirror the reference's flat module names so that its ``model.py`` dispatch reads
the same: ``newsEncoders.LIME`` / ``newsEncoders.CROWN`` / ``userEncoders.CROWN`` / ``Model`` /
``util.compute_scores``.  All arithmetic happens in ``liblime_b200.so`` (C ABI in
``include/lime_b200.h``); importing the package does not need a GPU, calling it does.
"""
from . import _lib
from . import attn_modules as layers
from . import news_modules as newsEncoders
from . import user_modules as userEncoders
from . import engine, ops, recommend, synth, trainer, training, util
from .model import Model
from .util import (NewsVectorCache, build_news_cache, compute_scores, evaluate_impressions,
                   score_impressions)

__all__ = ["Model", "newsEncoders", "userEncoders", "layers", "util", "engine", "ops", "recommend", "synth", "trainer", "training",
           "NewsVectorCache", "build_news_cache", "compute_scores", "evaluate_impressions",
           "score_impressions"]
