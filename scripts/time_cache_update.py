"""GPU: live news-vector cache updates (util.extend_news_cache) against a full rebuild, and the row-write kernel alone.

    python scripts/time_cache_update.py [--news 65238] [--ns 1,16,256,4096] [--modes fp32,bf16,fp32x3] [--reps 5] [--out FILE]

Workload: bench.py's MIND-shaped corpus (synth.make_news_table(65238, vocabulary 40,000)) and 4,096 further news drawn
the same way.  One JSON line per encoder mode and kind:
  build       util.build_news_cache over the corpus (host clock around a device synchronise, median of reps after a
              warm-up build)
  extend      util.extend_news_cache by n news into the corpus' cache, inside its headroom ("growth": false) and into a
              copy of it without headroom, so that every buffer is reallocated ("growth": true; the caching allocator
              is emptied before each such call, so every growth pays its cudaMalloc as a first growth does); host clock
              around a device synchronise, median of reps after a warm-up call; share_of_build = extend_ms / build_ms
  write_rows  lime_cache_write_rows alone over every row of the cache (CUDA events; 1.87 GB moved at 65,238 rows, far
              beyond the 126 MB L2), alternated in the same process with the derivation it replaced (split_candidates +
              news_meta + interleave_vg); achieved bytes/s and its fraction of the 7.7 TB/s data-sheet HBM bandwidth
The GPU name and power limit are read in the same process.
"""
import argparse
import dataclasses
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import lime_cikm25_b200 as L  # noqa: E402
from lime_cikm25_b200 import engine, ops, synth, util  # noqa: E402
from lime_cikm25_b200.config import default_config  # noqa: E402

ROW_BYTES = (852 + 1720) * 4 + (852 + 1720 + 8 + 800) * 4 + 2400 * 2     # read hist + cand, write all five roles
HBM_BYTES_PER_S = 7.7e12


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["sm_max_clock"] = [x.strip() for x in q.split(",")]
    except (OSError, ValueError, subprocess.TimeoutExpired):
        info["power_limit"] = "unavailable"
    return info


def host_ms(fn, prepare, reps):
    """Median host time of fn() from a synchronised device to a synchronised device; prepare() runs untimed before each."""
    out = []
    for _ in range(reps + 1):                     # the first call is the warm-up
        prepare()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        out.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(out[1:]))


def truncate(model, cache, n):
    """Back to the first n rows, inside the same buffers (undoes an extend between timed calls)."""
    cache._set_rows(n, cache.cand16.shape[0] - cache.news_num)
    util._write_tail(model, cache)


def without_headroom(model, cache):
    """A copy of the cache whose buffers hold exactly its rows: the next extend reallocates."""
    bufs = tuple(a.clone() for a in (cache.hist_rows, cache.cand_rows, cache.cand16, cache.meta, cache.hist_vg))
    c = util.NewsVectorCache(None, None, fingerprint=cache.fingerprint, buffers=bufs)
    c._set_rows(cache.news_num, cache.cand16.shape[0] - cache.news_num)
    return c


def events_ms(fn, reps, inner=5):
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--news", type=int, default=65238)
    ap.add_argument("--ns", default="1,16,256,4096")
    ap.add_argument("--modes", default="fp32,bf16,fp32x3")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_cache_update.py measures the GPU path: no CUDA device")
    info = gpu_info()
    cfg = default_config(vocabulary_size=40000, batch_size=32, word_embedding_init="skip")
    model = L.Model(cfg)
    model.initialize()
    synth.synthetic_parameters(model, seed=0)
    model = model.cuda().eval()
    news = synth.make_news_table(args.news, vocabulary_size=40000, seed=1)
    ns = [int(x) for x in args.ns.split(",")]
    extra = synth.make_news_table(max(ns), vocabulary_size=40000, seed=5)
    out = open(args.out, "a") if args.out else None

    def emit(line):
        line.update(info)
        print(json.dumps(line), flush=True)
        if out:
            out.write(json.dumps(line) + "\n")
            out.flush()

    eng = model.news_encoder.engine
    cache = None
    with torch.no_grad():
        for mode in args.modes.split(","):
            eng.bf16, eng.x3 = mode == "bf16", mode == "fp32x3"
            del cache
            cache = None
            holder = {}
            build_ms = host_ms(lambda: holder.update(c=util.build_news_cache(model, news)), lambda: holder.clear(), args.reps)
            cache = holder.pop("c")
            N = cache.news_num
            emit({"kind": "build", "mode": mode, "news": N, "ms": round(build_ms, 3), "capacity": cache.capacity})
            for n in ns:
                add = util_rows(extra, n)
                ms = host_ms(lambda: util.extend_news_cache(model, cache, add), lambda: truncate(model, cache, N), args.reps)
                emit({"kind": "extend", "mode": mode, "news": N, "n": n, "growth": False, "ms": round(ms, 4),
                      "share_of_build": round(ms / build_ms, 5)})
                copies = {}
                ms_g = host_ms(lambda: util.extend_news_cache(model, copies["c"], add),
                               lambda: (copies.update(c=without_headroom(model, cache)), torch.cuda.empty_cache()), args.reps)
                assert copies["c"].capacity > N
                del copies
                emit({"kind": "extend", "mode": mode, "news": N, "n": n, "growth": True, "ms": round(ms_g, 4),
                      "share_of_build": round(ms_g / build_ms, 5)})
            truncate(model, cache, N)
        # the write kernel alone, alternated with the derivation it replaced, on the last mode's rows
        se = model.scoring
        hist, cand = cache.hist_rows.clone(), cache.cand_rows.clone()
        dst = util.NewsVectorCache(None, None, buffers=tuple(torch.empty_like(a) for a in (
            cache.hist_rows, cache.cand_rows, cache.cand16, cache.meta, cache.hist_vg)))
        dst._set_rows(N, cache.cand16.shape[0] - N)
        ids = torch.arange(N, device="cuda")
        new = lambda: ops.cache_write_rows(hist, cand, ids, dst.hist_rows, dst.cand_rows, dst.cand16, dst.meta, dst.hist_vg)

        def old():
            c16 = se.split_candidates(cand)
            se.news_meta(hist, cand)
            engine.interleave_vg(hist)
            return c16
        new()
        old()
        t_new, t_old = [], []
        for _ in range(args.reps):
            t_new.append(events_ms(new, 3))
            t_old.append(events_ms(old, 3))
        k_ms, o_ms = float(np.median(t_new)), float(np.median(t_old))
        emit({"kind": "write_rows", "rows": N, "bytes": N * ROW_BYTES, "ms": round(k_ms, 4),
              "gb_per_s": round(N * ROW_BYTES / (k_ms * 1e-3) / 1e9, 1),
              "fraction_of_hbm": round(N * ROW_BYTES / (k_ms * 1e-3) / HBM_BYTES_PER_S, 3),
              "old_derivation_ms": round(o_ms, 4), "speedup_vs_old": round(o_ms / k_ms, 2)})


def util_rows(news, n):
    """The first n real news of a table (row 0 is its pad row), as a table of new news."""
    return dataclasses.replace(news, **{f: getattr(news, f)[1:n + 1] for f in
                                        ("title_text", "title_mask", "body_text", "body_mask", "category", "subCategory")})


if __name__ == "__main__":
    main()
