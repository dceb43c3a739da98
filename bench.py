#!/usr/bin/env python
"""bench.py — headline benchmark of the LIME scoring hot path (BASELINE.json configs[1]).

A *step* = one full evaluation pass over one impression set: fused scoring of every
(impression, candidate) pair on the cached news vectors, per-impression stable ranking and
AUC / MRR / nDCG@5 / nDCG@10, and (N > 1) the NCCL all-reduce of the five metric partial sums.
Metric: impressions/s (whole job).  See DESIGN.md "Measurement" for every definition used here.

  python bench.py --gpus N --steps K --warmup W            our arm (CUDA, sm_100a)
  python bench.py --impl reference ...                      the reference's algorithm on host cores
  python bench.py ... --dump-outputs DIR                    also write the last timed step's outputs as DIR/*.npy
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (it may be read-only)

import numpy as np
import torch

# The contract is ONE JSON line on stdout, but libraries write there too (NCCL prints "NCCL version ..." on the first
# communicator): file descriptor 1 is pointed at stderr for the whole run and the line goes to the saved descriptor.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(obj):
    os.write(_REAL_STDOUT, (json.dumps(obj) + "\n").encode())


METRIC = "eval_impressions_per_sec"
UNIT = "impressions/s"
D, H = 400, 50


def parse_args():
    a = _parse_args()
    if a.news is None:
        a.news = 73844 if a.shape == "adressa" else 65238
    return a


def _parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--shape", default="mind", choices=["mind", "adressa"],
                    help="synthetic data shape: MIND (default, BASELINE.json configs[1]) or Adressa (configs[3]: 73,844 news with "
                         "full 128-token bodies and short titles, 601,215 users)")
    ap.add_argument("--news", type=int, default=None, help="news in the vector cache (MIND: 65,238; Adressa: 73,844)")
    ap.add_argument("--vocab", type=int, default=40000)
    ap.add_argument("--impressions", type=int, default=73152, help="impressions per step per GPU (MIND-small dev size)")
    ap.add_argument("--batch-size", type=int, default=32, help="reference mini-batch size (GraphSAGE prefix)")
    ap.add_argument("--cpu-pairs", type=int, default=192, help="pairs in the bounded cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--bf16-encoder", action="store_true", help="run the 4 transformer GEMMs on tcgen05 (bf16 mode)")
    ap.add_argument("--encoder", default=None, choices=["fp32", "fp32x3", "bf16"],
                    help="Stage A mode of the scored cache: fp32 (FFMA, default), fp32x3 (tensor cores on fp16 hi/lo pairs, fp32-level accuracy), bf16")
    ap.add_argument("--train-steps", type=int, default=4, help="timed training steps of the secondary train_step report (0 = skip)")
    ap.add_argument("--train-batch", type=int, default=32, help="samples per rank per training step (BASELINE.json configs[2])")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: every rank scores its own --impressions set; strong: ONE set of --impressions is sharded over the "
                         "ranks by parallel.shard_impressions (balanced by sum(H + C))")
    ap.add_argument("--parity-impressions", type=int, default=12, help="impressions of the sampled fp64-oracle check (0 = skip)")
    ap.add_argument("--ref-cuda-batches", type=int, default=6, help="mini-batches of the reference-algorithm-on-CUDA leg (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (rank 0) as DIR/<name>.npy: scores [pairs] fp32, "
                         "per_impression_metrics [impressions, 4] and metric_sums [5] fp64; at most 64 MB in all.  "
                         "--impl reference: logits [batch, 1] fp32 of the last timed mini-batch")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


DUMP_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """Writes each array as <path>/<name>.npy.  If they hold more than DUMP_BYTES, every array larger than 1 MB keeps a
    fixed, seeded sample of its rows (sorted) and <name>_rows.npy records which rows, so that two runs with the same
    arguments write the same elements.  A <name>_rows.npy left in DIR by an earlier, sampled run is removed when <name>
    is written whole."""
    os.makedirs(path, exist_ok=True)
    big = [k for k, a in arrays.items() if a.nbytes > 1 << 20]
    room = DUMP_BYTES - sum(a.nbytes for k, a in arrays.items() if k not in big) - 2 * len(arrays) * 1024   # .npy headers
    out = dict(arrays)
    if sum(arrays[k].nbytes for k in big) > room:
        frac = room / sum(arrays[k].nbytes + 8 * len(arrays[k]) for k in big)
        for k in big:
            rows = np.sort(np.random.default_rng(0).choice(len(arrays[k]), size=int(len(arrays[k]) * frac), replace=False))
            out[k], out[k + "_rows"] = arrays[k][rows], rows.astype(np.float64)
    for k, a in out.items():
        np.save(os.path.join(path, k + ".npy"), a)
    for k in arrays:
        stale = os.path.join(path, k + "_rows.npy")
        if k + "_rows" not in out and os.path.exists(stale):
            os.remove(stale)


def algorithmic_bytes(imp):
    """SURVEY.md §8(d): per impression (H + C)(D*4 + 4 + 4 + 4 + 8) + H + 4C bytes (fp32)."""
    C = np.diff(imp.cand_off).astype(np.float64)
    return float(np.sum((H + C) * (D * 4 + 20) + H + 4 * C))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.kill)     # the sampler never outlives the benchmark, even one that fails
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].startswith("Active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def make_setup(args, rank, need_news_text=True, world=1):
    from lime_cikm25_b200 import synth
    from lime_cikm25_b200.config import default_config as make_config
    cfg = make_config(vocabulary_size=args.vocab, batch_size=args.batch_size, word_embedding_init="skip")
    if args.shape == "adressa":      # README.md:15 of the reference: title mean 6.63, bodies always truncated to the full 128 tokens
        news = synth.make_news_table(args.news, vocabulary_size=args.vocab, seed=1, body_full=True, title_mean=6.63)
        imp = synth.make_impressions(args.impressions, news.news_num, num_users=601215, seed=100 + rank)
    else:
        news = synth.make_news_table(args.news, vocabulary_size=args.vocab, seed=1)
        imp = synth.make_impressions(args.impressions, news.news_num, seed=100 + (0 if args.scaling == "strong" else rank))
    return cfg, news, imp


def cpu_baseline(args, cfg, news, imp, model_sd, steps=None, warmup=0):
    """The reference's algorithm (oracle port: per-pair batches, 51 news encodes per pair,
    util.py:88-112) on the host cores, on a bounded sample of the same workload: the first full mini-batches of the
    impression set, --cpu-pairs pairs of them, or exactly warmup + steps batches when steps is given."""
    from oracle import lime_oracle as O
    from lime_cikm25_b200 import synth
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    bs = args.batch_size
    batches = []
    for b in synth.impressions_to_pair_batches(news, imp, bs):      # a generator: only the batches taken are built
        if len(b[0]) == bs:
            batches.append(b)
        if len(batches) * bs >= (args.cpu_pairs if steps is None else bs * (steps + warmup)):
            break
    if steps is not None and len(batches) < steps + warmup:
        raise SystemExit("bench.py: the impression set holds %d full mini-batches of %d pairs, fewer than --warmup + --steps = %d"
                         % (len(batches), bs, steps + warmup))
    cbar = float(np.mean(np.diff(imp.cand_off)))
    times = []
    with torch.no_grad():
        for i, b in enumerate(batches):
            t0 = time.perf_counter()
            logits = O.model_forward(model_sd, b, cfg)
            times.append(time.perf_counter() - t0)
    timed = times[warmup:] if len(times) > warmup else times
    pairs_s = bs * len(timed) / sum(timed)
    return {"value": pairs_s / cbar, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "%d mini-batches of %d (user,candidate) pairs, each pair re-encoding %d news as "
                      "util.py:88-112 does; %.1f pairs/s; converted with mean %.1f candidates/impression"
                      % (len(timed), bs, H + 1, pairs_s, cbar),
            "pairs_per_sec": pairs_s, "ms_per_step": 1e3 * sum(timed) / len(timed), "last_logits": logits}


def run_reference(args):
    """--impl reference: rank 0 times the oracle port of the reference's CPU path."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import lime_cikm25_b200 as L
    from lime_cikm25_b200 import synth
    cfg, news, imp = make_setup(args, 0)
    model = L.Model(cfg)
    model.initialize()
    synth.synthetic_parameters(model, seed=0)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    steps = max(1, args.steps)            # one step = one reference mini-batch of 32 pairs (about 1 s on 16 cores)
    warm = max(1, args.warmup)
    cb = cpu_baseline(args, cfg, news, imp, sd, steps=steps, warmup=warm)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"logits": cb["last_logits"].numpy()})
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": cb["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, imp),
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def ref_cuda_leg(args, cfg, news, imp, model_sd, dev):
    """The reference's ALGORITHM on the GPU: the oracle port (same op sequence as the reference's PyTorch modules, one
    (user, candidate) pair per sample, 51 news encodes per pair, util.py:88-112 batching) with every tensor on the
    device -- the stand-in for 'the reference's own PyTorch CUDA eval throughput' of the north star (the reference itself
    cannot be installed: no packaging, absent dependencies; DESIGN.md section 5)."""
    from oracle import lime_oracle as O
    from lime_cikm25_b200 import synth
    bs = args.batch_size
    sd = {k: v.to(dev) for k, v in model_sd.items()}
    batches = []
    for b in synth.impressions_to_pair_batches(news, imp.slice(0, min(imp.num_impressions, 64)), bs):
        if len(b[0]) == bs:
            batches.append([torch.as_tensor(x).to(dev) for x in b])
        if len(batches) >= args.ref_cuda_batches + 2:
            break
    cbar = float(np.mean(np.diff(imp.cand_off)))
    try:
        with torch.no_grad():
            for b in batches[:2]:
                O.model_forward(sd, b, cfg)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for b in batches[2:]:
                O.model_forward(sd, b, cfg)
            e1.record()
            torch.cuda.synchronize()
        n = len(batches) - 2
        pairs_s = bs * n / (e0.elapsed_time(e1) * 1e-3)
        return {"value": pairs_s / cbar, "unit": UNIT, "pairs_per_sec": pairs_s, "kind": "port-on-cuda",
                "sample": "%d mini-batches of %d pairs, each pair re-encoding %d news (torch eager fp32 on the device)" % (n, bs, H + 1)}
    except Exception as e:      # the oracle is written for CPU tensors; report instead of failing the bench line
        return {"value": None, "unit": UNIT, "kind": "port-on-cuda", "error": "%s: %s" % (type(e).__name__, str(e)[:200])}


def parity_sample(args, model, cfg, cache, news, imp, model_sd, scores, dev):
    """Checker on the headline configuration itself: a few impressions' scores from the timed kernel vs the fp64 CPU
    oracle of the user encoder + click score evaluated on the same cached LIME vectors (Stage B in isolation)."""
    from oracle import lime_oracle as O
    se = model.scoring
    rng = np.random.default_rng(7)
    pick = np.sort(rng.choice(imp.num_impressions, size=min(args.parity_impressions, imp.num_impressions), replace=False))
    Hh = imp.hist_news.shape[1]
    sd64 = model_sd          # the oracle casts every weight to the dtype it is asked for (fp64 below)
    worst, npairs = 0.0, 0
    tail_start = (imp.num_pairs // args.batch_size) * args.batch_size
    got_all = scores.cpu().numpy()
    ref_all, got_sel = [], []
    for i in pick:
        hn = torch.as_tensor(imp.hist_news[i]).long()
        hv = se.lime_vectors(cache.hist_rows[hn.to(dev)], torch.as_tensor(imp.hist_fresh[i]).to(dev),
                             torch.as_tensor(imp.hist_life[i]).to(dev)).cpu().double()
        for p in range(int(imp.cand_off[i]), int(imp.cand_off[i + 1])):
            cn = int(imp.cand_news[p])
            cv = se.lime_vectors(cache.hist_rows[cn:cn + 1], torch.as_tensor(imp.cand_fresh[p:p + 1]).to(dev),
                                 torch.as_tensor(imp.cand_life[p:p + 1]).to(dev)).cpu().double()
            prefix = args.batch_size if p < tail_start else max(1, imp.num_pairs - tail_start)
            u = O.crown_user(sd64, hv.view(1, Hh, -1), torch.as_tensor(news.category[hn]).view(1, Hh),
                             torch.as_tensor(news.subCategory[hn]).view(1, Hh), torch.as_tensor(news.category[cn:cn + 1]).view(1, 1),
                             torch.as_tensor(news.subCategory[cn:cn + 1]).view(1, 1), torch.as_tensor(imp.hist_mask[i]).view(1, Hh),
                             cv.view(1, 1, -1), cfg, dtype=torch.float64, prefix_len=prefix)
            r = torch.tensor(float(np.float32(imp.cand_life[p]) - np.float32(imp.cand_fresh[p])))
            ref_all.append(float((u * cv.view(1, 1, -1)).sum() * O.lifetime_weight(r, cfg)))
            got_sel.append(float(got_all[p]))
            npairs += 1
    ref, got = np.asarray(ref_all), np.asarray(got_sel)
    floor = 0.1 * float(np.sqrt(np.mean(ref * ref))) + 1e-30
    worst = float(np.max(np.abs(got - ref) / np.maximum(np.abs(ref), floor)))
    return {"impressions": int(len(pick)), "pairs": npairs, "max_rel": worst, "tolerance": 1e-4,
            "oracle": "fp64 CPU oracle of userEncoders.CROWN.forward + RemainingLifetimeWeighting on the cached LIME vectors"}


def workload_config(args, imp):
    C = np.diff(imp.cand_off)
    name = ("Adressa-shaped eval (BASELINE.json configs[3]; full 128-token bodies)" if args.shape == "adressa"
            else "MIND-large-shaped eval (BASELINE.json configs[1])")
    return {"workload": "%s: %d-news fp32 vector cache, impression scoring + AUC/MRR/nDCG@5/10" % (name, args.news),
            "news": args.news, "impressions_per_step_per_gpu": imp.num_impressions,
            "pairs_per_step_per_gpu": int(imp.num_pairs), "history": H, "mean_candidates": float(C.mean()),
            "max_candidates": int(C.max()), "reference_batch_size": args.batch_size, "num_buckets": 10,
            "l2": "inputs exceed L2: the news-vector cache alone is %.0f MB vs 126 MB" % (args.news * (2572 * 4 + 2400 * 2 + 32) / 1e6)}


def train_report(args, cfg, news, dev, rank, world, bf16=False):
    """Secondary measurement (BASELINE.json configs[2]): one optimisation step as trainer.py:89-148 does it —
    forward (B x (50 history + 5 candidates) news encodes), loss, backward, [NCCL gradient all-reduce], clip, Adam —
    on the differentiable B200 path, fp32, batch resident in HBM.  Returns a dict for the JSON line."""
    import lime_cikm25_b200 as L
    from lime_cikm25_b200 import _lib, autograd, synth
    from lime_cikm25_b200.trainer import Trainer
    import torch.distributed as dist
    lib = _lib.require_device()
    autograd.set_bf16(bf16)
    torch.manual_seed(0)
    model = L.Model(cfg)
    model.initialize()
    synth.synthetic_parameters(model, seed=0)
    model = model.to(dev).train()
    tr = Trainer(model, cfg)
    B = args.train_batch
    batch = [torch.as_tensor(x).to(dev) for x in synth.make_train_batch(news, B, seed=500 + rank)]
    for _ in range(2):
        tr.step(batch)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    lib.lime_launch_count_reset()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.train_steps):
        loss = tr.step(batch)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.train_steps
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    news_per_step = B * (H + 5)
    autograd.set_bf16(False)
    return {"metric": "train_samples_per_sec", "gemm_mode": "bf16: TMA + tcgen05 GEMMs for forward / dX / dW on bf16 operand images, mma.sync attention forward + backward (fp32 accumulate, fp32 master weights and activations)" if bf16 else "fp32 FFMA", "value": B * world / (ms * 1e-3), "unit": "samples/s", "ms_per_step": ms,
            "batch_per_gpu": B, "history": H, "candidates": 5, "dtype": "bf16" if bf16 else "f32", "dropout_rate": float(cfg.dropout_rate),
            "news_encodes_per_step_per_gpu": news_per_step, "loss": float(loss),
            "tflops": 3 * 241.3e6 * news_per_step / (ms * 1e-3) / 1e12,
            "gpu_launches_per_step": int(lib.lime_launch_count()) // max(1, args.train_steps),
            "allreduce_bytes_per_step": int(getattr(tr, "allreduce_bytes", 0)),
            "optimizer": "torch.optim.Adam + clip_grad_norm_(4.0), as trainer.py:33,147"}


def run_b200(args):
    import lime_cikm25_b200 as L
    from lime_cikm25_b200 import _lib, engine, parallel, synth, util
    import torch.distributed as dist

    rank, world, local = parallel.init_from_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    lib = _lib.require_device()
    cfg, news, imp = make_setup(args, rank, world=world)
    pair_base, total_pairs = 0, None
    if args.scaling == "strong" and world > 1:
        imp, pair_base, total_pairs = parallel.shard_impressions(imp, rank, world)
    model = L.Model(cfg)
    model.initialize()
    synth.synthetic_parameters(model, seed=0)
    sd_cpu = {k: v.detach().clone() for k, v in model.state_dict().items()} if rank == 0 else None
    model = model.to(dev).eval()
    enc_mode = args.encoder or ("bf16" if args.bf16_encoder else "fp32")
    eng = model.news_encoder.engine

    def set_mode(mode):
        eng.bf16, eng.x3 = mode == "bf16", mode == "fp32x3"

    # ---- news-vector cache (Stage A), built once per checkpoint; timed and reported separately ----
    with torch.no_grad():
        model.scoring.fold()
        # the other encoder modes first, timed only (the scored cache is the one selected by --encoder)
        other_modes = {}
        for mode in ("fp32", "fp32x3", "bf16"):
            if mode == enc_mode:
                continue
            set_mode(mode)
            for rep in range(2):          # the second build is the reported one: the first pays one-time setup (allocator growth, tensor-map encoder)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                other = util.build_news_cache(model, news, dev)
                torch.cuda.synchronize()
                other_modes[mode] = time.perf_counter() - t0
                del other
        set_mode(enc_mode)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        cache = util.build_news_cache(model, news, dev)
        torch.cuda.synchronize()
        cache_s = time.perf_counter() - t0
    dimp = engine.DeviceImpressions(imp, dev)
    torch.cuda.synchronize()
    scores = torch.empty(dimp.num_pairs, dtype=torch.float32, device=dev)
    bs = args.batch_size

    def step():
        return util.evaluate_device(model, cache, dimp, bs, pair_base, total_pairs, scores_out=scores, want_ranks=False,
                                    sharded=world > 1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.no_grad():
        for _ in range(max(3, args.warmup)):
            step()
        barrier()
        # ---- timed region: exactly K steps, CUDA events on the launching stream, max over ranks ----
        sampler = ClockSampler(local) if rank == 0 else None
        lib.lime_launch_count_reset()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            last_scores, _, last_per_imp, sums = step()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        launches = int(lib.lime_launch_count())
        result = sums.tolist()
        if args.dump_outputs and rank == 0:      # before the passes below reuse the scores buffer
            dump_outputs(args.dump_outputs, {"scores": last_scores.cpu().numpy(),
                                             "per_impression_metrics": last_per_imp.cpu().numpy(),
                                             "metric_sums": sums.cpu().numpy()})
        fallback_units = int(dimp.work_counter[1])      # units of the last timed step that the exact kernel re-scored
        # ---- the dominant kernel alone (roofline numerator) ----
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record()
        for _ in range(args.steps):
            util.score_impressions(model, cache, dimp, bs, pair_base, total_pairs, out=scores)
        k1.record()
        torch.cuda.synchronize()
        kernel_ms = k0.elapsed_time(k1) / args.steps
        # ---- end to end: host (pinned) inputs -> H2D -> score -> metrics -> D2H of the 5 sums, EVERY step ----
        # Two device copies of the impression arrays: the upload of step i + 1 (copy stream) overlaps the kernels of
        # step i, as an evaluation loop over successive impression sets does; every step still copies all its inputs
        # from pinned host memory and reads its result back.
        dimp_b = engine.DeviceImpressions(imp, dev)
        bufs = [dimp, dimp_b]
        main_stream, copy_stream = torch.cuda.current_stream(), torch.cuda.Stream()
        ev_up = [torch.cuda.Event(), torch.cuda.Event()]
        ev_done = [torch.cuda.Event(), torch.cuda.Event()]

        def e2e_step_fn(d):
            return util.evaluate_device(model, cache, d, bs, pair_base, total_pairs, scores_out=scores, want_ranks=False,
                                        sharded=world > 1)

        barrier()
        t0 = time.perf_counter()
        with torch.cuda.stream(copy_stream):
            bufs[0].upload()
            ev_up[0].record(copy_stream)
        for i in range(args.steps):
            cur = i & 1
            main_stream.wait_event(ev_up[cur])
            sums_i = e2e_step_fn(bufs[cur])[3]
            ev_done[cur].record(main_stream)
            if i + 1 < args.steps:
                with torch.cuda.stream(copy_stream):
                    if i >= 1:
                        copy_stream.wait_event(ev_done[cur ^ 1])     # the kernels of step i - 1 no longer read that buffer
                    bufs[cur ^ 1].upload()
                    ev_up[cur ^ 1].record(copy_stream)
            s = sums_i.tolist()                                      # device -> host read of the step's result
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        assert abs(s[0] - result[0]) <= 1e-9 * max(1.0, abs(result[0])), "e2e path disagrees with the resident path"
        clocks = sampler.stop() if sampler else None
        parity = ref_cuda = None
        if rank == 0 and world == 1:
            util.score_impressions(model, cache, dimp, bs, pair_base, total_pairs, out=scores)
            torch.cuda.synchronize()
            if args.parity_impressions > 0:
                parity = parity_sample(args, model, cfg, cache, news, imp, sd_cpu, scores, dev)
            if args.ref_cuda_batches > 0:
                ref_cuda = ref_cuda_leg(args, cfg, news, imp, sd_cpu, dev)

    train = None
    if args.train_steps > 0:
        del cache, scores
        torch.cuda.empty_cache()
        train = train_report(args, cfg, news, dev, rank, world, bf16=True)
        train["fp32"] = {k: v for k, v in train_report(args, cfg, news, dev, rank, world, bf16=False).items()
                         if k in ("value", "ms_per_step", "tflops", "loss", "gemm_mode")}

    t = torch.tensor([ms, e2e_s * 1e3], dtype=torch.float64, device=dev)
    tot = torch.tensor([dimp.num_impressions, dimp.num_pairs], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms, e2e_ms = t.tolist()
    total_imp, total_pairs_all = tot.tolist()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (burst copy)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    alg = algorithmic_bytes(imp)
    achieved = alg / (kernel_ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "score_traffic.json")
    if os.path.isfile(tpath):
        tj = json.load(open(tpath))
        w = tj.get("workload", {})
        if w.get("news") == args.news and w.get("impressions") == args.impressions and w.get("history") == H:
            traffic = float(tj["dram_bytes_read"]) + float(tj["dram_bytes_write"])
    line = {
        "metric": METRIC, "value": total_imp * args.steps / (ms * 1e-3), "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": args.scaling if world > 1 else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, imp),
        "pairs_per_sec": total_pairs_all * args.steps / (ms * 1e-3),
        "e2e": {"value": total_imp * args.steps / (e2e_ms * 1e-3), "unit": UNIT,
                "h2d_bytes_per_step": dimp.h2d_bytes(), "d2h_bytes_per_step": 40,
                "overlap": "H2D of step i+1 (copy stream, second device buffer) overlaps the kernels of step i",
                "cache_build_included": False,
                "note": "per-step inputs are the impression arrays; the news-vector cache is per checkpoint (cache_build, eval_wall_one_checkpoint)"},
        "eval_wall_one_checkpoint": {"seconds": cache_s + ms * 1e-3 / args.steps, "cache_build_s": cache_s, "scoring_step_s": ms * 1e-3 / args.steps,
                                     "what": "one checkpoint evaluated on one impression set: news-vector cache build + one eval step"},
        "fallback_units": fallback_units, "units_per_step_per_gpu": int(dimp.num_units),
        "gpu_launches": launches,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "kernel": "lime::score_tc_kernel", "kernel_ms": kernel_ms,
                     "algorithmic_bytes_per_launch": alg, "peak_source": peak_src,
                     "note": "kernel_ms = one lime_score_impressions call (score_tc_kernel + the usually empty exact-"
                             "fallback launch), CUDA events. traffic = ncu dram bytes of one launch (profiles/score_traffic.json): "
                             "a unique history row is read as vc|gw (3200 B), a candidate as fp16 hi/lo pairs of w1|w2|w3 (4800 B). "
                             "No pipe is saturated: the kernel is bound by the memory + barrier round trip of its 7 operand stages "
                             "per unit (DESIGN.md section 3)"},
        "clocks": clocks,
        "cache_build": {"seconds": cache_s, "news_per_sec": news.news_num / cache_s,
                        "tflops": news.news_num * 241.3e6 / cache_s / 1e12,
                        "encoder": enc_mode,
                        "other_modes": {mode: {"seconds": sec, "news_per_sec": news.news_num / sec, "tflops": news.news_num * 241.3e6 / sec / 1e12}
                                        for mode, sec in other_modes.items()},
                        "modes": "fp32 = FFMA kernels (reference-accurate default, 1e-4 vs the reference's vectors); fp32x3 = every dense layer "
                                 "one tcgen05 launch on fp16 hi/lo pairs (lo.hi + hi.lo and hi.hi in two TMEM accumulators), attention on mma.sync "
                                 "hi/lo pairs (vectors 3e-6 from the fp32 mode); bf16 = bf16 activations, TMA + tcgen05 GEMMs, tensor-core attention "
                                 "(metrics within 1e-3); other_modes: second of two builds"},
        "metrics": {"auc": result[0] / result[4], "mrr": result[1] / result[4],
                    "ndcg5": result[2] / result[4], "ndcg10": result[3] / result[4]},
    }
    if parity is not None:
        line["parity_sample"] = parity
    if ref_cuda is not None:
        line["ref_cuda"] = ref_cuda
        if ref_cuda.get("value"):
            line["vs_ref_cuda"] = line["e2e"]["value"] / ref_cuda["value"]
    if train is not None:
        line["train_step"] = train
    if world == 1 and not args.no_cpu_baseline:
        cb = cpu_baseline(args, cfg, news, imp, sd_cpu)
        line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
