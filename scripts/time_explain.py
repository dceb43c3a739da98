"""GPU: recommend.explain of the top_k(10) lists of U users beside recommend.top_k itself, one JSON line per history length.

    python scripts/time_explain.py [--users 8192] [--histories 50,200] [--k 10] [--reps 5] [--out FILE]

Workload: the 65,238-news cache of bench.py's MIND shape (BASELINE.json configs[1]) and a pool of every news, freshness /
lifetime drawn as in scripts/time_recommend.py; U histories of H slots from synth.make_impressions.  Per H:
  topk_ms        recommend.top_k(k) over all U users (scores every pool news, keeps k), synchronised
  explain_ms     recommend.explain of those [U, k] lists (exact kernel, k pairs per user, every output at full size)
  explain_share  explain_ms / topk_ms
The two calls alternate in the same process, each timed with CUDA events around the call after one warm-up of both,
and the median of ``reps`` runs is reported.  The GPU name and power limit are read in the same process.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import lime_cikm25_b200 as L  # noqa: E402
from lime_cikm25_b200 import recommend, synth, util  # noqa: E402
from lime_cikm25_b200.config import default_config  # noqa: E402
from time_recommend import gpu_info, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--news", type=int, default=65238)
    ap.add_argument("--users", type=int, default=8192)
    ap.add_argument("--histories", default="50,200")
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_explain.py measures the GPU path: no CUDA device")
    info = gpu_info()
    cfg = default_config(vocabulary_size=40000, batch_size=32, word_embedding_init="skip")
    model = L.Model(cfg)
    model.initialize()
    synth.synthetic_parameters(model, seed=0)
    model = model.cuda().eval()
    news = synth.make_news_table(args.news, vocabulary_size=40000, seed=1)
    rng = np.random.default_rng(3)
    C = news.news_num - 1
    pool_news = np.arange(1, news.news_num, dtype=np.int32)
    pool_fresh = np.exp(rng.uniform(0.0, np.log(1e7), C)).astype(np.float32)
    pool_life = np.exp(rng.uniform(np.log(600.0), np.log(6e5), C)).astype(np.float32)
    out = open(args.out, "a") if args.out else None
    with torch.no_grad():
        cache = util.build_news_cache(model, news, "cuda")
        plan = recommend.plan(model, cache, pool_news, pool_fresh, pool_life)
        for H in (int(h) for h in args.histories.split(",")):
            imp = synth.make_impressions(args.users, news.news_num, max_history=H, seed=2)
            hist = [torch.from_numpy(np.ascontiguousarray(a)).cuda()
                    for a in (imp.hist_news, imp.hist_mask.astype(np.uint8), imp.hist_fresh, imp.hist_life)]
            tk = lambda: recommend.top_k(model, cache, plan, *hist, args.k)
            res = tk()                                                                            # warm-up
            ex = lambda: recommend.explain(model, cache, plan, *hist, res.news)
            e = ex()
            t_topk, t_ex = [], []
            for _ in range(args.reps):                                                            # alternated
                t_topk.append(timed(tk, 1))
                t_ex.append(timed(ex, 1))
            ok = res.news >= 0
            d = (e.score[ok].double() - res.score[ok].double()).abs().max().item()
            topk_ms, ex_ms = float(np.median(t_topk)), float(np.median(t_ex))
            line = dict(kind="explain", users=args.users, history=H, k=args.k, pool=C, pairs_explained=int(ok.sum()),
                        topk_ms=round(topk_ms, 2), explain_ms=round(ex_ms, 2), explain_share=round(ex_ms / topk_ms, 5),
                        topk_ms_runs=[round(x, 2) for x in t_topk], explain_ms_runs=[round(x, 2) for x in t_ex],
                        max_abs_score_diff_vs_topk=d, users_per_explain_batch=max(1, min(args.users, recommend.EXPLAIN_BUDGET // (args.k * (3 * H + 3)))),
                        **info)
            print(json.dumps(line), flush=True)
            if out:
                out.write(json.dumps(line) + "\n")
                out.flush()
    if out:
        out.close()


if __name__ == "__main__":
    main()
