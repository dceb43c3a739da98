"""End-to-end parity of the CUDA path with (a) the golden vectors produced by the unmodified
reference and (b) the CPU oracle, through the drop-in module API and the C ABI.

Logit tolerance: 1e-4 relative (north star), measured as max|a-b| / max(|b|, 0.1*rms(b)) — see
tests/test_oracle_golden.py::rel for why a floor is needed; integer work (buckets, ranks) is exact.
"""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import lime_cikm25_b200 as L  # noqa: E402
from lime_cikm25_b200 import engine, ops, parallel, synth, util  # noqa: E402
from oracle import lime_oracle as O  # noqa: E402
from oracle.make_golden import CASES, case_inputs  # noqa: E402
from oracle.ref_import import make_config  # noqa: E402

DEV = "cuda"
TOL = 1e-4


def rel(a, b, floor=None):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    if floor is None:
        floor = 0.1 * float(np.sqrt(np.mean(b * b))) + 1e-30
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), floor)))


def load_case(case, golden_dir, **cfg_over):
    spec, cfg, news, imp = case_inputs(case)
    g = np.load(os.path.join(golden_dir, case + ".npz"))
    cfg.word_embedding_init = "skip"
    for k, v in cfg_over.items():
        setattr(cfg, k, v)
    model = L.Model(cfg)
    model.initialize()
    checksum = synth.synthetic_parameters(model, spec["weights_seed"])
    assert checksum == float(g["weights_checksum"]), "synthetic weights were not regenerated identically"
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    return cfg, news, imp, g, sd, model.to(DEV).eval()


@pytest.mark.parametrize("case", ["small_bs8", "buckets20"])
def test_news_encoder_stage_vectors(lib, case, golden_dir):
    """CROWN.forward -> 900-d content and LIME.forward -> 400-d vectors vs the reference's outputs."""
    cfg, news, imp, g, sd, model = load_case(case, golden_dir)
    n0 = g["content"].shape[0]
    t = lambda a: torch.as_tensor(a[:n0]).unsqueeze(0).to(DEV)
    fresh, life = torch.as_tensor(g["stage_fresh"]).to(DEV), torch.as_tensor(g["stage_life"]).to(DEV)
    args = (t(news.title_text), t(news.title_mask), t(news.title_text) * 0, t(news.body_text), t(news.body_mask),
            t(news.body_text) * 0, t(news.category), t(news.subCategory), None)
    with torch.no_grad():
        content = model.news_encoder.base_news_encoder(*args, None, None)[0]
        vec = model.news_encoder(*args, fresh.unsqueeze(0), life.unsqueeze(0))[0]
    assert content.shape == (n0, 900) and vec.shape == (n0, 400)
    assert rel(content.cpu().numpy(), g["content"]) < TOL
    assert rel(vec.cpu().numpy(), g["lime_vec"]) < TOL
    # the cache's two-part representation reproduces the same vector
    hist, cand = model.scoring.build_rows(*(x[0].contiguous() for x in (args[0], args[3], args[6], args[7])))
    assert rel(model.scoring.lime_vectors(hist, fresh, life).cpu().numpy(), g["lime_vec"]) < TOL


@pytest.mark.parametrize("case", ["small_bs8", "buckets20"])
def test_news_encoder_fp32x3_mode_matches_reference(lib, case, golden_dir):
    """fp32x3 mode (every transformer GEMM as three tensor-core passes on fp16 hi / lo operand pairs, 2^-21 per product): the
    encoder outputs meet the same 1e-4 bar against the reference's vectors as the fp32 FFMA mode (measured worst element 1.9e-5
    vs 9.6e-6).  It stays opt-in because the scoring stage amplifies the difference: with it as the default, one logit of
    test_bucket_sweep_and_flags leaves the 1e-4 bar."""
    cfg, news, imp, g, sd, model = load_case(case, golden_dir)
    n0 = g["content"].shape[0]
    t = lambda a: torch.as_tensor(a[:n0]).to(DEV).contiguous()
    fresh, life = torch.as_tensor(g["stage_fresh"]).to(DEV), torch.as_tensor(g["stage_life"]).to(DEV)
    model.news_encoder.engine.x3 = True
    try:
        with torch.no_grad():
            content = model.news_encoder.engine.encode_content(t(news.title_text), t(news.body_text), t(news.category), t(news.subCategory))
            hist, cand = model.scoring.build_rows(t(news.title_text), t(news.body_text), t(news.category), t(news.subCategory))
        assert rel(content.cpu().numpy(), g["content"]) < TOL
        assert rel(model.scoring.lime_vectors(hist, fresh, life).cpu().numpy(), g["lime_vec"]) < TOL
    finally:
        model.news_encoder.engine.x3 = False


@pytest.mark.parametrize("case", sorted(CASES))
def test_model_forward_matches_reference(lib, case, golden_dir):
    """Model.forward on the reference's own eval mini-batches (26 tensors, one pair per sample)."""
    cfg, news, imp, g, sd, model = load_case(case, golden_dir)
    out = []
    with torch.no_grad():
        for batch in synth.impressions_to_pair_batches(news, imp, cfg.batch_size):
            tb = [torch.as_tensor(x).to(DEV) for x in batch]
            logits = model(*tb, tb[24] - tb[23])
            assert logits.shape == (len(batch[0]), 1)
            out.append(logits.squeeze(1).cpu())
    scores = torch.cat(out).numpy()
    assert np.array_equal(scores == 0, g["scores"] == 0)           # saturated weights give exact zeros
    assert rel(scores, g["scores"]) < TOL


@pytest.mark.parametrize("case", sorted(CASES))
def test_cached_impression_eval_matches_reference(lib, case, golden_dir):
    """News-vector cache + impression-major scoring + device ranking/metrics == compute_scores."""
    cfg, news, imp, g, sd, model = load_case(case, golden_dir)
    with torch.no_grad():
        cache = util.build_news_cache(model, news)
        dimp = engine.DeviceImpressions(imp, DEV)
        metrics, det = util.evaluate_impressions(model, cache, dimp, cfg.batch_size, return_details=True)
    scores = det["scores"].cpu().numpy()
    assert np.array_equal(scores == 0, g["scores"] == 0)
    assert rel(scores, g["scores"]) < TOL
    assert np.allclose(metrics, g["metrics"], atol=1e-3)
    # ranks: exact unless two non-tied reference scores are closer than the fp32 tolerance
    ranks = det["ranks"].cpu().numpy()
    want = np.concatenate(O.evaluate_impressions(
        [scores[imp.cand_off[i]:imp.cand_off[i + 1]] for i in range(imp.num_impressions)],
        [imp.labels[imp.cand_off[i]:imp.cand_off[i + 1]] for i in range(imp.num_impressions)])[1])
    assert np.array_equal(ranks, want)
    assert (ranks != g["ranks"]).mean() < 0.1
    # base score (no lifetime weighting) exposes every pair un-saturated
    model.config.use_remaining_lifetime_weighting = False
    with torch.no_grad():
        base = util.score_impressions(model, cache, dimp, cfg.batch_size).cpu().numpy()
    assert rel(base, g["base_scores"]) < TOL


def _reference_style_forward(model, tb):
    """model.py:158-181 spelled out over the plugin classes: unsqueeze the candidate tensors (eval), news_encoder ->
    user_encoder -> remaining_lifetime_weighting.  tb = the 25 dataset tensors on the device."""
    (uid, ucat, usub, utt, utm, ute, uct, ucm, uce, ufr, ulf, umask, ugraph, ucmask, ucidx,
     ncat, nsub, ntt, ntm, nte, nct, ncm, nce, nfr, nlf) = tb
    rem = nlf - nfr
    if ncat.dim() == 1:
        ncat, nsub, ntt, ntm, nct, ncm, nte, nce, nfr, nlf, rem = (x.unsqueeze(1) for x in (ncat, nsub, ntt, ntm, nct, ncm, nte, nce, nfr, nlf, rem))
    news_rep = model.news_encoder(ntt, ntm, nte, nct, ncm, nce, ncat, nsub, None, news_freshness=nfr, news_user_topic_lifetime=nlf)
    user_rep = model.user_encoder(utt, utm, ute, uct, ucm, uce, ncat, nsub, ucat, usub, umask, ugraph, ucmask, ucidx, None,
                                  news_rep, user_freshness=ufr, user_user_topic_lifetime=ulf)
    assert user_rep.shape == news_rep.shape
    return model.remaining_lifetime_weighting(user_rep, news_rep, rem)


@pytest.mark.parametrize("case", ["small_bs8", "bs64"])
def test_plugin_classes_compose_like_reference_model(lib, case, golden_dir):
    """The plugin classes are real modules: news_encoder -> userEncoders.CROWN.forward -> [B,N,D] ->
    RemainingLifetimeWeighting.forward, composed as the reference's model.py:171-181 does, reproduce the reference's
    scores (P < H and P > H cases), and agree with this package's fused Model.forward."""
    cfg, news, imp, g, sd, model = load_case(case, golden_dir)
    out, fused = [], []
    with torch.no_grad():
        for batch in synth.impressions_to_pair_batches(news, imp, cfg.batch_size):
            tb = [torch.as_tensor(x).to(DEV) for x in batch]
            logits = _reference_style_forward(model, tb)
            assert logits.shape == (len(batch[0]), 1)
            out.append(logits.squeeze(1).cpu())
            fused.append(model(*tb, tb[24] - tb[23]).squeeze(1).cpu())
    scores = torch.cat(out).numpy()
    assert rel(scores, g["scores"]) < TOL
    assert rel(scores, torch.cat(fused).numpy()) < TOL


def test_reference_model_py_over_plugin_classes(lib, golden_dir):
    """INTEGRATION.md section A variant 1, literally: the reference's own model.py with its newsEncoders / userEncoders /
    util imports resolved to this package.  Needs /root/reference (build container) AND a GPU: skipped elsewhere."""
    from oracle import ref_import
    if not ref_import.reference_available():
        pytest.skip("reference tree not present (GPU box)")
    cfg, news, imp, g, sd, model = load_case("small_bs8", golden_dir)
    ref_model = ref_import.load_reference_model_over_plugins().Model(cfg)
    missing, unexpected = ref_model.load_state_dict(sd, strict=False)
    assert not unexpected and all(k.endswith("pe") for k in missing), (missing, unexpected)
    ref_model = ref_model.to(DEV).eval()
    out = []
    with torch.no_grad():
        for batch in synth.impressions_to_pair_batches(news, imp, cfg.batch_size):
            tb = [torch.as_tensor(x).to(DEV) for x in batch]
            out.append(ref_model(*tb, tb[24] - tb[23]).squeeze(1).cpu())
    assert rel(torch.cat(out).numpy(), g["scores"]) < TOL


def _stage_b_oracle(model, sd, cfg, cache, news, imp, prefix, dtype=torch.float32, remaining=None):
    """CPU oracle of the user encoder + click score on the GPU-built LIME vectors (isolates Stage B):
    O.score_from_vectors per impression.  ``prefix``: the GraphSAGE prefix, an int or one per pair [P];
    ``remaining``: the pairs' remaining lifetime [P] (default: life - freshness in fp32, as the callers derive it)."""
    se = model.scoring
    out = np.zeros(imp.num_pairs, np.float64 if dtype == torch.float64 else np.float32)
    pre = np.broadcast_to(np.asarray(prefix, np.int64), (imp.num_pairs,))
    rem = imp.cand_life - imp.cand_fresh if remaining is None else np.asarray(remaining, np.float32)
    for i in range(imp.num_impressions):
        p0, p1 = int(imp.cand_off[i]), int(imp.cand_off[i + 1])
        if p1 == p0:
            continue
        hn = torch.as_tensor(imp.hist_news[i]).long()
        cn = torch.as_tensor(imp.cand_news[p0:p1]).long()
        hv = se.lime_vectors(cache.hist_rows[hn.to(DEV)], torch.as_tensor(imp.hist_fresh[i]).to(DEV),
                             torch.as_tensor(imp.hist_life[i]).to(DEV)).cpu()
        cv = se.lime_vectors(cache.hist_rows[cn.to(DEV)], torch.as_tensor(imp.cand_fresh[p0:p1]).to(DEV),
                             torch.as_tensor(imp.cand_life[p0:p1]).to(DEV)).cpu()
        hn_, cn_ = imp.hist_news[i], imp.cand_news[p0:p1]
        out[p0:p1] = O.score_from_vectors(sd, cfg, hv, news.category[hn_], news.subCategory[hn_], imp.hist_mask[i], cv,
                                          news.category[cn_], news.subCategory[cn_], rem[p0:p1], pre[p0:p1], dtype).numpy()
    return out


@pytest.mark.parametrize("H,cand,prefix", [(200, 70, 32), (100, 5, 120), (20, 300, 7), (50, 1, 64), (223, 40, 100)])
def test_scoring_kernel_sweep_shapes(lib, H, cand, prefix):
    """Sweep shapes of BASELINE.json configs[4]: history up to 223 (multi-chunk register tiling),
    300 candidates (multi-unit impressions), GraphSAGE prefix below / above H.  The exact kernel and the
    default mode (cache operands passed: tensor cores, chunked beyond 56 slots) against the fp64 reference."""
    cfg = make_config(vocabulary_size=400, batch_size=128, max_history_num=H, word_embedding_init="skip")
    model = L.Model(cfg)
    model.initialize()
    synth.synthetic_parameters(model, 5)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    model = model.to(DEV).eval()
    news = synth.make_news_table(90, vocabulary_size=400, seed=H)
    imp = synth.make_impressions(2, news.news_num, max_history=H, cand_fixed=cand, near_zero_frac=0.9, seed=cand)
    imp.hist_mask[1, H // 2:] = False
    with torch.no_grad():
        cache = util.build_news_cache(model, news)
        dimp = engine.DeviceImpressions(imp, DEV)
        got = model.scoring.score(cache.hist_rows, cache.cand_rows, dimp, prefix_main=prefix).cpu().numpy()
        tc = model.scoring.score(cache.hist_rows, cache.cand_rows, dimp, prefix_main=prefix, cand16=cache.cand16, meta=cache.meta,
                                 hist_vg=cache.hist_vg).cpu().numpy()
        want = _stage_b_oracle(model, sd, cfg, cache, news, imp, prefix, torch.float64)
    assert rel(got, want) < TOL and rel(tc, want) < TOL


def test_bucket_sweep_and_flags(lib):
    """B = 50 buckets (2,500-entry tables) and the weighting flags of util.py:34-46."""
    for over in (dict(num_buckets=50), dict(use_expired_penalty=False), dict(use_remaining_lifetime_weighting=False)):
        cfg = make_config(vocabulary_size=300, batch_size=8, word_embedding_init="skip", **over)
        model = L.Model(cfg)
        model.initialize()
        synth.synthetic_parameters(model, 6)
        sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
        model = model.to(DEV).eval()
        news = synth.make_news_table(40, vocabulary_size=300, seed=1)
        imp = synth.make_impressions(3, news.news_num, cand_fixed=4, near_zero_frac=0.8, seed=2)
        with torch.no_grad():
            cache = util.build_news_cache(model, news)
            got = util.score_impressions(model, cache, engine.DeviceImpressions(imp, DEV), 8).cpu().numpy()
            want = O.score_pairs_reference_style(sd, news, imp, cfg, 8).numpy()
        assert rel(got, want) < TOL, over


def test_properties_at_scale(lib):
    """Size-independent properties on a MIND-shaped run too large for the CPU oracle: determinism,
    invariance to the unit tiling and to rank sharding, rank permutations, metric ranges."""
    cfg = make_config(vocabulary_size=5000, batch_size=32, word_embedding_init="skip")
    model = L.Model(cfg)
    model.initialize()
    synth.synthetic_parameters(model, 7)
    model = model.to(DEV).eval()
    news = synth.make_news_table(3000, vocabulary_size=5000, seed=11)
    imp = synth.make_impressions(4000, news.news_num, seed=12)
    with torch.no_grad():
        cache = util.build_news_cache(model, news)
        cache2 = util.build_news_cache(model, news, chunk=700)
        assert torch.equal(cache.hist_rows, cache2.hist_rows) and torch.equal(cache.cand_rows, cache2.cand_rows)
        d52 = engine.DeviceImpressions(imp, DEV)    # default tile
        d13 = engine.DeviceImpressions(imp, DEV, tile_c=16)
        m1, det1 = util.evaluate_impressions(model, cache, d52, 32, return_details=True)
        m2, det2 = util.evaluate_impressions(model, cache, d52, 32, return_details=True)
        s13 = util.score_impressions(model, cache, d13, 32)
    assert torch.equal(det1["scores"], det2["scores"]) and m1 == m2                 # deterministic
    # tiling-invariant: the interpolation nodes depend on the unit's candidates, so not bit-for-bit
    assert rel(s13.cpu().numpy(), det1["scores"].cpu().numpy()) < 1e-5
    # the tensor-core path agrees with the exact per-pair kernel, and forcing every unit through the
    # fallback list reproduces the exact kernel bit for bit
    try:
        with torch.no_grad():
            ops.score_configure(ops.SCORE_EXACT)
            s_exact = util.score_impressions(model, cache, d52, 32).clone()
            ops.score_configure(ops.SCORE_FORCE_FALLBACK)
            s_forced = util.score_impressions(model, cache, d52, 32).clone()
    finally:
        ops.score_configure(ops.SCORE_AUTO)
    assert torch.equal(s_exact, s_forced)
    assert rel(det1["scores"].cpu().numpy(), s_exact.cpu().numpy()) < 2e-5
    assert float((det1["scores"] - s_exact).abs().max()) > 0                       # two different kernels ran
    assert all(0.0 <= x <= 1.0 for x in m1)
    ranks = det1["ranks"].cpu().numpy()
    for i in range(0, imp.num_impressions, 97):
        r = np.sort(ranks[imp.cand_off[i]:imp.cand_off[i + 1]])
        assert np.array_equal(r, np.arange(1, len(r) + 1))                           # a permutation of 1..C
    # 4-way impression sharding (what 4 ranks would do) reproduces scores bit-for-bit and the means
    sums = torch.zeros(5, dtype=torch.float64, device=DEV)
    parts = []
    with torch.no_grad():
        for r in range(4):
            sub, base, total = parallel.shard_impressions(imp, r, 4)
            d = engine.DeviceImpressions(sub, DEV)
            _, det = util.evaluate_impressions(model, cache, d, 32, pair_index_base=base, total_pairs=total,
                                               return_details=True)
            parts.append(det["scores"])
            sums += det["sums"]
    assert torch.equal(torch.cat(parts), det1["scores"])
    assert np.allclose((sums[:4] / sums[4]).cpu().numpy(), m1, atol=1e-12)
    # scores do not depend on the order of the candidates inside an impression
    perm = imp.slice(0, 50)
    order = np.concatenate([np.arange(perm.cand_off[i], perm.cand_off[i + 1])[::-1] for i in range(50)])
    flipped = synth.Impressions(perm.hist_news, perm.hist_mask, perm.hist_fresh, perm.hist_life, perm.cand_off,
                                perm.cand_news[order], perm.cand_fresh[order], perm.cand_life[order],
                                perm.labels[order], perm.user_id)
    with torch.no_grad():
        a = model.scoring.score(cache.hist_rows, cache.cand_rows, engine.DeviceImpressions(perm, DEV), 32)
        b = model.scoring.score(cache.hist_rows, cache.cand_rows, engine.DeviceImpressions(flipped, DEV), 32)
    assert rel(b.cpu().numpy(), a[torch.as_tensor(order).to(DEV)].cpu().numpy()) < 1e-5


def test_dedup_of_repeated_history_rows(lib):
    """The tensor-core kernel merges history slots with equal (news, bucket pair, mask) into one operand row with a
    multiplicity.  Exercise every way the multiplicity enters: repeated clicked news inside the unmasked part (both
    attention softmaxes, pooling), the same news with a different bucket pair or a different mask (must NOT merge),
    a history that is one single row, and GraphSAGE prefixes that cut through a run of equal slots (main and tail)."""
    H = 50
    cfg = make_config(vocabulary_size=400, batch_size=32, max_history_num=H, word_embedding_init="skip")
    model = L.Model(cfg)
    model.initialize()
    synth.synthetic_parameters(model, 11)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    model = model.to(DEV).eval()
    news = synth.make_news_table(120, vocabulary_size=400, seed=3)
    imp = synth.make_impressions(4, news.news_num, max_history=H, cand_fixed=9, near_zero_frac=0.5, seed=17)
    imp.hist_mask[:] = True
    # impression 0: slots 3, 4, 17, 40 are the same click (same news, same ages); slot 41 the same news, other ages
    for h in (4, 17, 40, 41):
        imp.hist_news[0, h] = imp.hist_news[0, 3]
    for h in (4, 17, 40):
        imp.hist_fresh[0, h], imp.hist_life[0, h] = imp.hist_fresh[0, 3], imp.hist_life[0, 3]
    imp.hist_fresh[0, 41], imp.hist_life[0, 41] = 5e6, 700.0
    # impression 1: the masked tail repeats a clicked (news, ages) pair: equal keys except for the mask
    imp.hist_mask[1, 30:] = False
    imp.hist_news[1, 30:] = imp.hist_news[1, 2]
    imp.hist_fresh[1, 30:], imp.hist_life[1, 30:] = imp.hist_fresh[1, 2], imp.hist_life[1, 2]
    # impression 2: the whole history is one row
    imp.hist_news[2, :] = imp.hist_news[2, 0]
    imp.hist_fresh[2, :], imp.hist_life[2, :] = imp.hist_fresh[2, 0], imp.hist_life[2, 0]
    # impression 3: short history, zero padding (the common case)
    imp.hist_mask[3, 6:] = False
    imp.hist_news[3, 6:] = 0
    imp.hist_fresh[3, 6:] = 0
    imp.hist_life[3, 6:] = 0
    model.config.use_remaining_lifetime_weighting = False
    try:
        with torch.no_grad():
            cache = util.build_news_cache(model, news)
            dimp = engine.DeviceImpressions(imp, DEV)
            want = _stage_b_oracle(model, sd, cfg, cache, news, imp, 5)
            out = {}
            for name, mode in (("tc", ops.SCORE_AUTO), ("exact", ops.SCORE_EXACT)):
                ops.score_configure(mode, 1e-6)
                out[name] = model.scoring.score(cache.hist_rows, cache.cand_rows, dimp, prefix_main=5, cand16=cache.cand16,
                                                meta=cache.meta).cpu().numpy()
                assert int(dimp.work_counter[1]) == 0            # nothing handed to the fallback
                # the last 13 pairs form a short mini-batch of the reference: prefix 4 cuts the run of slots 3, 4
                out[name + "_tail"] = model.scoring.score(cache.hist_rows, cache.cand_rows, dimp, prefix_main=18,
                                                          tail_start=imp.num_pairs - 13, prefix_tail=4, cand16=cache.cand16,
                                                          meta=cache.meta).cpu().numpy()
    finally:
        ops.score_configure(ops.SCORE_AUTO, 1e-6)
    assert rel(out["tc"], want) < TOL and rel(out["exact"], want) < TOL
    assert rel(out["tc"], out["exact"]) < 5e-5 and rel(out["tc_tail"], out["exact_tail"]) < 5e-5
    assert np.abs(out["tc_tail"] - out["tc"]).max() > 1e-4        # the prefix really matters on this data


def test_split_f16_pairs_and_news_meta(lib):
    """Cache-build helpers of the tensor-core path: x * 1024 = hi + lo to 2^-21, layout [hi | lo][k][400] (an operand-row
    triple = 3 consecutive 800-byte rows); the meta sector repeats the cached topic id / bounds / folded scalars."""
    g = torch.Generator().manual_seed(5)
    x = (torch.randn(37, 1720, generator=g) * torch.logspace(-4, 1, 1720)).to(DEV)
    x[5, 7] = 0.0
    stamp = torch.zeros(37, device=DEV)
    pairs = ops.split_f16_pairs(x, 3, absmax=stamp)
    assert pairs.dtype == torch.float16 and pairs.shape == (37, 2400)
    p = pairs.double().view(37, 2, 3, 400)
    back = (p[:, 0] + p[:, 1]).reshape(37, 1200) / 1024.0
    ref = x[:, :1200].double()
    # 2^-21 relative; values below 1e-4 put their lo half into the fp16 subnormals (6e-8 resolution / 1024)
    assert bool(((back - ref).abs() <= 2.0 ** -20 * ref.abs() + 1e-10).all())
    assert torch.equal(stamp, x[:, :1200].abs().max(dim=1).values)


def test_compute_scores_drop_in(lib, tmp_path, monkeypatch):
    """util.compute_scores with the reference's signature: rank file + truth file round trip."""
    import types
    cfg = make_config(vocabulary_size=300, batch_size=8, word_embedding_init="skip", category_lifetime_map=None)
    model = L.Model(cfg)
    model.initialize()
    synth.synthetic_parameters(model, 8)
    model = model.to(DEV)
    news = synth.make_news_table(40, vocabulary_size=300, seed=3)
    imp = synth.make_impressions(9, news.news_num, cand_mean=5, near_zero_frac=0.5, seed=4)
    beh, idx = [], []
    for i in range(imp.num_impressions):
        n = int(imp.hist_mask[i].sum())
        for p in range(imp.cand_off[i], imp.cand_off[i + 1]):
            beh.append([int(imp.user_id[i]), imp.hist_news[i].tolist(), imp.hist_mask[i].copy(), int(imp.cand_news[p]),
                        i, float(imp.cand_fresh[p]), float(imp.cand_life[p]), imp.hist_fresh[i, :n].tolist(),
                        imp.hist_life[i, :n].tolist()])
            idx.append(i)
    corpus = types.SimpleNamespace(
        dev_behaviors=beh, dev_indices=idx, max_history_num=50,
        config=types.SimpleNamespace(vocabulary_size=300, category_num=18, subCategory_num=270),
        news_title_text=news.title_text, news_title_mask=news.title_mask, news_abstract_text=news.body_text,
        news_abstract_mask=news.body_mask, news_category=news.category, news_subCategory=news.subCategory)
    monkeypatch.chdir(tmp_path)
    os.makedirs("dev/ref")
    with open("dev/ref/truth-small.txt", "w") as f:
        for i in range(imp.num_impressions):
            lab = imp.labels[imp.cand_off[i]:imp.cand_off[i + 1]].tolist()
            f.write(("" if i == 0 else "\n") + str(i + 1) + " " + str(lab).replace(" ", ""))
    res = str(tmp_path / "res.txt")
    metrics = util.compute_scores(model, corpus, 8, "dev", res, "small")
    sd = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}
    want_scores = O.score_pairs_reference_style(sd, news, imp, cfg, 8).numpy()
    want, ranks = O.evaluate_impressions(
        [want_scores[imp.cand_off[i]:imp.cand_off[i + 1]] for i in range(imp.num_impressions)],
        [imp.labels[imp.cand_off[i]:imp.cand_off[i + 1]] for i in range(imp.num_impressions)])
    assert np.allclose(metrics, want, atol=1e-3)
    lines = open(res).read().split("\n")
    assert len(lines) == imp.num_impressions and lines[0].startswith("1 [")


def test_bf16_mode_metrics(lib, golden_dir):
    """bf16 mode (north star): the four transformer GEMMs of the news encoder on tcgen05 with bf16
    operands; AUC/MRR/nDCG@5/10 within 1e-3 absolute of the fp32 path, stage vectors bf16-accurate."""
    cfg, news, imp, g, sd, model = load_case("small_bs8", golden_dir)
    n0 = g["content"].shape[0]
    t = lambda a: torch.as_tensor(a[:n0]).to(DEV).contiguous()
    model.news_encoder.engine.bf16 = True
    with torch.no_grad():
        content = model.news_encoder.engine.encode_content(t(news.title_text), t(news.body_text), t(news.category),
                                                           t(news.subCategory))
    c = content.cpu().numpy().astype(np.float64)
    rms = float(np.sqrt(np.mean((c - g["content"]) ** 2)) / np.sqrt(np.mean(g["content"].astype(np.float64) ** 2)))
    assert 1e-6 < rms < 1e-2, rms        # bf16-accurate, and the tensor-core path really ran (not bit-equal to fp32)

    cfg = make_config(vocabulary_size=5000, batch_size=32, word_embedding_init="skip")
    model = L.Model(cfg)
    model.initialize()
    synth.synthetic_parameters(model, 7)
    model = model.to(DEV).eval()
    news = synth.make_news_table(2500, vocabulary_size=5000, seed=21)
    imp = synth.make_impressions(3000, news.news_num, seed=22)
    res = {}
    with torch.no_grad():
        dimp = engine.DeviceImpressions(imp, DEV)
        for mode in (False, True):
            model.news_encoder.engine.bf16 = mode
            cache = util.build_news_cache(model, news)
            res[mode] = util.evaluate_impressions(model, cache, dimp, 32)
    assert np.allclose(res[True], res[False], atol=1e-3), (res[True], res[False])


def test_tensor_core_scoring_paths(lib):
    """Every branch of lime_score_impressions on one impression set: expansion units (default tolerance), a tolerance
    below the expansion's remainder bound (those units are re-scored by the exact kernel in the same call), all
    units through the exact-fallback list (tolerance 0), exact kernel only; edge impressions: empty history
    (uniform attention), one candidate (zero-width interval), 300 candidates (9 units), and operands beyond the
    fp16 range (flagged for the exact kernel)."""
    cfg = make_config(vocabulary_size=600, batch_size=32, word_embedding_init="skip")
    model = L.Model(cfg)
    model.initialize()
    synth.synthetic_parameters(model, 9)
    model = model.to(DEV).eval()
    news = synth.make_news_table(400, vocabulary_size=600, seed=31)
    imp = synth.make_impressions(60, news.news_num, seed=32)
    imp.hist_mask[0, :] = False                                     # empty history
    imp.hist_news[0, :] = 0
    imp.hist_mask[1, 1:] = False                                    # a single clicked news
    edge = [synth.make_impressions(1, news.news_num, cand_fixed=c, seed=40 + c) for c in (1, 2, 300)]
    def cat(a, b):
        off = np.concatenate([a.cand_off, b.cand_off[1:] + a.cand_off[-1]])
        return synth.Impressions(np.concatenate([a.hist_news, b.hist_news]), np.concatenate([a.hist_mask, b.hist_mask]),
                                 np.concatenate([a.hist_fresh, b.hist_fresh]), np.concatenate([a.hist_life, b.hist_life]), off,
                                 np.concatenate([a.cand_news, b.cand_news]), np.concatenate([a.cand_fresh, b.cand_fresh]),
                                 np.concatenate([a.cand_life, b.cand_life]), np.concatenate([a.labels, b.labels]),
                                 np.concatenate([a.user_id, b.user_id]))
    for e in edge:
        imp = cat(imp, e)
    model.config.use_remaining_lifetime_weighting = False           # every pair un-saturated
    out, fallback = {}, {}
    try:
        with torch.no_grad():
            cache = util.build_news_cache(model, news)
            dimp = engine.DeviceImpressions(imp, DEV)
            for name, (mode, tol) in dict(two=(ops.SCORE_AUTO, 1e-6), tight=(ops.SCORE_AUTO, 1e-13), forced=(ops.SCORE_FORCE_FALLBACK, 1e-6),
                                          exact=(ops.SCORE_EXACT, 1e-6)).items():
                ops.score_configure(mode, tol)
                out[name] = util.score_impressions(model, cache, dimp, 32).clone()
                fallback[name] = int(dimp.work_counter[1])
            # operands outside the fp16 range: scale one history news' cached vectors beyond 32768
            big = cache.hist_rows.clone()
            big[int(imp.hist_news[2, 0]), :400] *= 1e6
            ops.score_configure(ops.SCORE_AUTO, 1e-6)
            s_big = model.scoring.score(big, cache.cand_rows, dimp, prefix_main=32).clone()
            fb_big = int(dimp.work_counter[1])
            ops.score_configure(ops.SCORE_EXACT, 1e-6)
            s_big_exact = model.scoring.score(big, cache.cand_rows, dimp, prefix_main=32).clone()
    finally:
        ops.score_configure(ops.SCORE_AUTO, 1e-6)
    ex = out["exact"].cpu().numpy()
    assert fallback["two"] == 0 and 0 < fallback["tight"] <= dimp.num_units and fallback["forced"] == dimp.num_units
    assert torch.equal(out["forced"], out["exact"])
    assert rel(out["two"].cpu().numpy(), ex) < 5e-5 and rel(out["tight"].cpu().numpy(), ex) < 5e-5
    assert float((out["two"] - out["tight"]).abs().max()) > 0       # expansion vs exact re-scoring: different code paths
    assert fb_big >= 1                                              # flagged, re-scored exactly
    users = [i for i in range(imp.num_impressions) if int(imp.hist_news[2, 0]) in imp.hist_news[i]]
    sel = np.concatenate([np.arange(imp.cand_off[i], imp.cand_off[i + 1]) for i in users])
    assert torch.equal(s_big[sel], s_big_exact[sel])
    assert np.isfinite(s_big.cpu().numpy()).all()


@pytest.mark.parametrize("H,prefix", [(100, 32), (200, 32), (112, 130), (200, 103), (224, 57), (64, 40)])
def test_long_history_on_the_tensor_core_path(lib, H, prefix):
    """H > 56 (BASELINE.json configs[4]): the history is cut into chunks of <= 56 slots, the attention weights over the FULL
    history come from a pre-pass, every chunk runs on the tensor-core kernel and the partial pooling states are merged
    (lime_score_impressions_long).  Same scores as the exact per-pair kernel and as the fp64 reference, no unit handed to the
    fallback; ragged histories, a masked tail, multi-unit impressions and GraphSAGE prefixes that end inside chunk 1
    (H = 64, 224) or chunk 2 (H = 200, prefix 103), or lie above H, included."""
    from lime_cikm25_b200 import ops
    cfg = make_config(vocabulary_size=400, batch_size=128, max_history_num=H, word_embedding_init="skip")
    model = L.Model(cfg)
    model.initialize()
    synth.synthetic_parameters(model, 5)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    model = model.to(DEV).eval()
    news = synth.make_news_table(300, vocabulary_size=400, seed=H)
    imp = synth.make_impressions(40, news.news_num, max_history=H, cand_mean=30.0, near_zero_frac=0.3, seed=H + 1)
    imp.hist_mask[1, H // 2:] = False
    imp.hist_mask[2, :] = False
    with torch.no_grad():
        cache = util.build_news_cache(model, news)
        dimp = engine.DeviceImpressions(imp, DEV)
        got = model.scoring.score(cache.hist_rows, cache.cand_rows, dimp, prefix_main=prefix, cand16=cache.cand16, meta=cache.meta,
                                  hist_vg=cache.hist_vg).cpu().numpy()
        assert dimp.chunked(cfg.num_buckets) is not None and int(dimp.work_counter[1]) == 0
        ops.score_configure(ops.SCORE_EXACT, 1e-6)
        try:
            want = model.scoring.score(cache.hist_rows, cache.cand_rows, engine.DeviceImpressions(imp, DEV), prefix_main=prefix,
                                       cand16=cache.cand16, meta=cache.meta, hist_vg=cache.hist_vg).cpu().numpy()
        finally:
            ops.score_configure(ops.SCORE_AUTO, 1e-6)
        ref = _stage_b_oracle(model, sd, cfg, cache, news, imp, prefix, torch.float64)
    assert rel(got, want) < 5e-5
    assert rel(got, ref) < TOL and rel(want, ref) < TOL
