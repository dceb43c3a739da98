"""Pin the CPU oracle (oracle/lime_oracle.py) against the golden vectors produced by running the
unmodified reference (oracle/make_golden.py).  No GPU."""
import os

import numpy as np
import pytest
import torch

import lime_cikm25_b200 as L
from lime_cikm25_b200 import synth
from oracle import lime_oracle as O
from oracle.make_golden import CASES, case_inputs


def load_case(case, golden_dir):
    spec, cfg, news, imp = case_inputs(case)
    g = np.load(os.path.join(golden_dir, case + ".npz"))
    cfg.word_embedding_init = "skip"
    model = L.Model(cfg)
    model.initialize()
    checksum = synth.synthetic_parameters(model, spec["weights_seed"])
    assert checksum == float(g["weights_checksum"]), "synthetic weights were not regenerated identically"
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    return spec, cfg, news, imp, g, sd


def rel(a, b, floor=None):
    """Parity metric for logits: max |a-b| / max(|b|, floor), floor = 0.1 * rms(b) by default.
    A pure per-element relative error is meaningless on near-cancelling logits: the reference's own
    fp32 result differs from the fp64 value of the same formula by 3e-3 of the logit where
    |logit| < 1e-3 * rms (measured on the bs64 fixture), while its error stays < 3e-6 * rms."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    if floor is None:
        floor = 0.1 * float(np.sqrt(np.mean(b * b))) + 1e-30
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), floor)))


@pytest.mark.parametrize("case", sorted(CASES))
def test_oracle_scores_match_reference(case, golden_dir):
    spec, cfg, news, imp, g, sd = load_case(case, golden_dir)
    torch.set_num_threads(os.cpu_count())
    with torch.no_grad():
        scores = O.score_pairs_reference_style(sd, news, imp, cfg, cfg.batch_size).numpy()
        cfg_nw = type(cfg)(**{**vars(cfg), "use_remaining_lifetime_weighting": False})
        base = O.score_pairs_reference_style(sd, news, imp, cfg_nw, cfg.batch_size).numpy()
    assert rel(base, g["base_scores"]) < 2e-5            # fp32 vs fp32, different op fusion
    assert np.array_equal(scores == 0, g["scores"] == 0)  # saturated weights: exact zeros agree
    assert rel(scores, g["scores"]) < 2e-5
    (auc, mrr, n5, n10), ranks = O.evaluate_impressions(
        [scores[imp.cand_off[i]:imp.cand_off[i + 1]] for i in range(imp.num_impressions)],
        [imp.labels[imp.cand_off[i]:imp.cand_off[i + 1]] for i in range(imp.num_impressions)])
    assert np.allclose([auc, mrr, n5, n10], g["metrics"], atol=1e-3)


@pytest.mark.parametrize("case", ["small_bs8", "buckets20"])
def test_oracle_stage_vectors_match_reference(case, golden_dir):
    spec, cfg, news, imp, g, sd = load_case(case, golden_dir)
    n0 = g["content"].shape[0]
    t = lambda a: torch.as_tensor(a[:n0])
    with torch.no_grad():
        content = O.crown_content(sd, t(news.title_text), t(news.body_text), t(news.category), t(news.subCategory), cfg)
        vec = O.lime_news(sd, t(news.title_text), t(news.body_text), t(news.category), t(news.subCategory),
                          torch.as_tensor(g["stage_fresh"]), torch.as_tensor(g["stage_life"]), cfg)
    assert rel(content.numpy(), g["content"]) < 2e-5
    assert rel(vec.numpy(), g["lime_vec"]) < 2e-5


def test_oracle_bucketize_bit_exact(golden_dir):
    g = np.load(os.path.join(golden_dir, "buckets.npz"))
    for nb in (10, 20, 50):
        got = O.bucketize(torch.as_tensor(g["x_%d" % nb]), nb).numpy()
        assert np.array_equal(got, g["b_%d" % nb])
    # the divisor the CUDA kernel hard-codes (csrc/common.cuh) is torch's fp32 log(86400)
    assert torch.log(torch.tensor(60 * 60 * 24.0)).view(torch.int32).item() == 0x4135DE2E


def test_oracle_ranks_and_metrics_match_reference(golden_dir):
    g = np.load(os.path.join(golden_dir, "metrics.npz"))
    off = g["cand_off"]
    s = [g["scores"][off[i]:off[i + 1]] for i in range(len(off) - 1)]
    y = [g["labels"][off[i]:off[i + 1]] for i in range(len(off) - 1)]
    m, ranks = O.evaluate_impressions(s, y)
    assert np.array_equal(np.concatenate(ranks), g["ranks"])      # stable, -0.0 == 0.0
    assert np.allclose(m, g["metrics"], rtol=0, atol=1e-12)


@pytest.mark.parametrize("case", ["small_bs8", "bs64"])
def test_score_from_vectors_reproduces_model_forward(case, golden_dir):
    """score_from_vectors (Stage B from LIME vectors, the fp64 reference of the scoring kernels) is model_forward's own
    user encoder + click score: fed model_forward's cand / hist parts, it gives the same logits, with the GraphSAGE
    prefix of the reference's mini-batch (the runtime batch size, shorter on the last batch).  In fp32 the two differ
    only by the batching of the same products (the oracle's own fp32-vs-fp32 bar); in fp64 they agree to rounding."""
    spec, cfg, news, imp, g, sd = load_case(case, golden_dir)
    for dtype, bar in ((torch.float32, 1e-5), (torch.float64, 1e-12)):
        got, want = [], []
        with torch.no_grad():
            for batch in synth.impressions_to_pair_batches(news, imp, cfg.batch_size):
                logits, parts = O.model_forward(sd, batch, cfg, dtype, return_parts=True)
                u_cat, u_sub, u_mask, n_cat, n_sub = (torch.as_tensor(np.asarray(batch[k])) for k in (1, 2, 11, 15, 16))
                B = logits.shape[0]
                for b in range(B):
                    got.append(O.score_from_vectors(sd, cfg, parts["hist"][b], u_cat[b], u_sub[b], u_mask[b], parts["cand"][b],
                                                    n_cat[b].view(1), n_sub[b].view(1), parts["remaining"][b].view(1), B, dtype))
                want.append(logits.view(-1))
        got, want = torch.cat(got).numpy(), torch.cat(want).numpy()
        assert got.dtype == want.dtype == {torch.float32: np.float32, torch.float64: np.float64}[dtype]
        assert np.array_equal(got == 0, want == 0)
        assert rel(got, want) < bar, (dtype, rel(got, want))
    assert rel(got, g["scores"]) < 1e-4            # fp64 against the reference's fp32 run: its own rounding only
