"""GPU: top-k recommendation over a news pool (recommend.plan / recommend.top_k), one JSON line per (pool, k), and its
full-pool evaluation (recommend.evaluate), one JSON line per pool ("kind": "evaluate").

    python scripts/time_recommend.py [--users 4096] [--pools all,16384,4096] [--ks 10,100] [--targets 8] [--out FILE]

Workload: the 65,238-news cache of bench.py's MIND shape (BASELINE.json configs[1]), U histories from
synth.make_impressions, a pool of every news or a random subset, freshness / lifetime drawn like synth's candidates.
Per configuration:
  plan_ms                 recommend.plan (host checks, sort, unit template, upload), synchronised
  score_ms_per_launch     lime_score_impressions over one batch of PAIR_BUDGET / C users, sorted plan
  score_ms_caller_order   the same batch with the pool in the caller's order, units cut by engine.build_units' rule for
                          caller-ordered candidates (candidates + distinct bucket pairs <= 40 operand-row triples);
                          the two plans alternate in the same process
  topk_ms_per_launch      lime_pool_topk on that batch's scores (clicked exclusion on), torch_topk_ms torch.topk on the
                          same tensor
  users_per_s             recommend.top_k over all U users, end to end (scores, selection, id mapping)
Evaluation, T targets per user drawn from the pool (cutoffs 10, 50, 100):
  rank_ms_per_launch      lime_pool_rank_metrics (memset + count + finish) on the batch topk_ms_per_launch uses
  rank_share_of_scoring   rank_ms_per_launch / score_ms_per_launch
  eval_users_per_s        recommend.evaluate over all U users, end to end, alternated in the same process with
                          recommend.top_k at k = 10 (topk_users_per_s)
All times are CUDA events after a warm-up of every shape; the GPU name and power limit are read in the same process.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import lime_cikm25_b200 as L  # noqa: E402
from lime_cikm25_b200 import engine, ops, recommend, synth, util  # noqa: E402
from lime_cikm25_b200.config import default_config  # noqa: E402


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["sm_max_clock"] = [x.strip() for x in q.split(",")]
    except (OSError, ValueError, subprocess.TimeoutExpired):
        info["power_limit"] = "unavailable"
    return info


def timed(fn, reps, inner=1):
    """Median over ``reps`` CUDA-event windows of ``inner`` back-to-back fn() calls, per call (ms).  inner > 1 for
    sub-millisecond calls: the device then runs the calls back to back instead of waiting for the host to issue each."""
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(inner):
            fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b) / inner)
    return float(np.median(out))


def caller_order_plan(model, cache, news, fresh, life):
    """The pool in the caller's order, units by build_units' greedy rule (the comparator of the sorted plan)."""
    p = recommend.plan(model, cache, news, fresh, life)
    dev = p.device
    C = news.size
    bp = engine._host_bucket_pairs(fresh, life, int(model.config.num_buckets))
    _, p0, cnt = engine.build_units(np.asarray([0, C]), engine.TC_TRIPLES - 2, bp, engine.TC_TRIPLES)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    q = engine.PoolPlan(news=d(news.astype(np.int32)), fresh=d(fresh), life=d(life), remaining=None,
                        index=torch.arange(C, dtype=torch.int32, device=dev), exclude=None, bucket_pair=d(bp),
                        topic=p.topic[torch.argsort(p.index.long())], caller_news=p.caller_news)
    q.templates[engine.TC_TRIPLES - 2] = (d(p0.astype(np.int32)), d(cnt.astype(np.int32)))
    return q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--news", type=int, default=65238)
    ap.add_argument("--users", type=int, default=4096)
    ap.add_argument("--pools", default="all,16384,4096")
    ap.add_argument("--ks", default="10,100")
    ap.add_argument("--targets", type=int, default=8, help="held-out clicks per user of the evaluation pass")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_recommend.py measures the GPU path: no CUDA device")
    info = gpu_info()
    cfg = default_config(vocabulary_size=40000, batch_size=32, word_embedding_init="skip")
    model = L.Model(cfg)
    model.initialize()
    synth.synthetic_parameters(model, seed=0)
    model = model.cuda().eval()
    news = synth.make_news_table(args.news, vocabulary_size=40000, seed=1)
    with torch.no_grad():
        cache = util.build_news_cache(model, news, "cuda")
    imp = synth.make_impressions(args.users, news.news_num, seed=2)
    hist = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (imp.hist_news, imp.hist_mask, imp.hist_fresh, imp.hist_life)]
    hist[1] = hist[1].to(torch.uint8)
    rng = np.random.default_rng(3)
    trng = np.random.default_rng(4)              # targets: a stream of their own, the pools stay those of rng
    out = open(args.out, "a") if args.out else None

    def emit(line):
        print(json.dumps(line), flush=True)
        if out:
            out.write(json.dumps(line) + "\n")
            out.flush()
    for pool_arg in args.pools.split(","):
        C = news.news_num - 1 if pool_arg == "all" else int(pool_arg)
        pool_news = (np.arange(1, news.news_num) if pool_arg == "all"
                     else rng.choice(np.arange(1, news.news_num), C, replace=False)).astype(np.int32)
        pool_fresh = np.exp(rng.uniform(0.0, np.log(1e7), C)).astype(np.float32)
        pool_life = np.exp(rng.uniform(np.log(600.0), np.log(6e5), C)).astype(np.float32)
        with torch.no_grad():
            plan = recommend.plan(model, cache, pool_news, pool_fresh, pool_life)                  # warm-up
            plan_ms = timed(lambda: recommend.plan(model, cache, pool_news, pool_fresh, pool_life), args.reps)
            plan = recommend.plan(model, cache, pool_news, pool_fresh, pool_life)
            caller = caller_order_plan(model, cache, pool_news, pool_fresh, pool_life)
            ub = max(1, min(args.users, recommend.PAIR_BUDGET // C))
            hb = [h[:ub] for h in hist]
            dimps = {name: engine.DeviceImpressions.from_pool(p, *hb) for name, p in (("sorted", plan), ("caller", caller))}
            scores = torch.empty(ub * C, dtype=torch.float32, device="cuda")

            def score(name):
                return model.scoring.score(cache.hist_rows, cache.cand_rows, dimps[name], prefix_main=cfg.batch_size, out=scores,
                                           cand16=cache.cand16, meta=cache.meta, hist_vg=cache.hist_vg)
            t = {"sorted": [], "caller": []}
            fb = {}
            for name in ("sorted", "caller"):
                score(name)                                                                       # warm-up
            for _ in range(args.reps):                                                            # alternated
                for name in ("sorted", "caller"):
                    t[name].append(timed(lambda: score(name), 1))
                    fb[name] = int(dimps[name].work_counter[1])
            score("sorted")
            s2 = scores.view(ub, C)
            for k in (int(x) for x in args.ks.split(",")):
                topk = lambda: ops.pool_topk(s2, k, plan.index, plan.news, None, hb[0], hb[1])
                ttk = lambda: torch.topk(s2, k, dim=1)
                topk(), ttk()
                topk_ms, torch_ms = timed(topk, args.reps, 20), timed(ttk, args.reps, 20)
                res = recommend.top_k(model, cache, plan, *hist, k)                              # warm-up of every batch shape
                e2e_ms = timed(lambda: recommend.top_k(model, cache, plan, *hist, k), max(1, args.reps // 2))
                res = recommend.top_k(model, cache, plan, *hist, k)
                line = dict(pool=C, users=args.users, k=k, users_per_launch=ub, plan_ms=round(plan_ms, 3),
                            score_ms_per_launch=round(float(np.median(t["sorted"])), 3),
                            score_ms_caller_order=round(float(np.median(t["caller"])), 3),
                            topk_ms_per_launch=round(topk_ms, 4), torch_topk_ms=round(torch_ms, 4),
                            topk_share_of_scoring=round(topk_ms / float(np.median(t["sorted"])), 5),
                            users_per_s=round(args.users / (e2e_ms / 1e3), 1), e2e_ms=round(e2e_ms, 2),
                            fallback_units=res.fallback_units, fallback_units_batch_sorted=fb["sorted"],
                            fallback_units_batch_caller=fb["caller"], units_per_user=int(plan.units(engine.TC_TRIPLES - 2)[0].numel()),
                            units_per_user_caller_order=int(caller.templates[engine.TC_TRIPLES - 2][0].numel()),
                            cache_news=news.news_num - 1, history=int(imp.hist_news.shape[1]), **info)
                emit(line)

            cutoffs = (10, 50, 100)
            tgt = torch.from_numpy(pool_news[trng.integers(0, C, (args.users, args.targets))]).cuda()
            tmask = torch.ones(tgt.shape, dtype=torch.bool, device="cuda")
            pos = plan.positions(cache.news_num)[tgt[:ub].long()].contiguous()
            rank = lambda: ops.pool_rank_metrics(s2, plan.index, pos, cutoffs, plan.news, None, hb[0], hb[1])
            rank()
            rank_ms = timed(rank, args.reps, 20)
            ev = lambda: recommend.evaluate(model, cache, plan, *hist, tgt, tmask, cutoffs=cutoffs)
            tk = lambda: recommend.top_k(model, cache, plan, *hist, 10)
            ev(), tk()                                                                            # warm-up
            te, tt = [], []
            for _ in range(max(1, args.reps // 2)):                                               # alternated
                te.append(timed(ev, 1))
                tt.append(timed(tk, 1))
            res = ev()
            score_ms = float(np.median(t["sorted"]))
            emit(dict(kind="evaluate", pool=C, users=args.users, targets=args.targets, cutoffs=list(cutoffs), users_per_launch=ub,
                      score_ms_per_launch=round(score_ms, 3), rank_ms_per_launch=round(rank_ms, 4),
                      rank_share_of_scoring=round(rank_ms / score_ms, 5),
                      eval_users_per_s=round(args.users / (float(np.median(te)) / 1e3), 1),
                      topk_users_per_s=round(args.users / (float(np.median(tt)) / 1e3), 1),
                      eval_e2e_ms=round(float(np.median(te)), 2), topk_e2e_ms=round(float(np.median(tt)), 2),
                      ranked_per_user=round(float(res.ranked.double().mean()), 3), fallback_units=res.fallback_units,
                      cache_news=news.news_num - 1, history=int(imp.hist_news.shape[1]), **info))
    if out:
        out.close()


if __name__ == "__main__":
    main()
