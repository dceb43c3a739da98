"""Parity of the bf16 modes against fp64 references that round to bf16 exactly where the kernels round
(tests/bf16_reference.py): the three tensor-core attention cores (mha_tc_kernel, mha_fwd_tc_kernel, mha_bwd_tc_kernel)
at their pass structures, odd head widths, strided layouts, sharp / flat softmax, dropout and the 65,535-news launch
boundary; the Stage A bf16 cache build's content vector; and the bf16 training step (encode_news, then one
model_forward step with dropout), its output and every parameter's gradient.

Every comparison also measures the kernel's distance to EXACT fp64 (no rounding) and asserts that the rounding reference
is at least 10x closer: otherwise the reference would not model the kernel.  Bars are about 3x the worst error measured
on a B200 (DESIGN.md section 4 lists the measured values)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import lime_cikm25_b200 as L  # noqa: E402
from lime_cikm25_b200 import ops, synth, training  # noqa: E402
from lime_cikm25_b200 import autograd as A  # noqa: E402
from bf16_reference import Bf16Attention, attention_exact, bf, bf16_attn, crown_content_bf16, mha_eval_bf16, train_mm  # noqa: E402
from test_gpu_training_parity import STEP_SEED, device_keep, oracle_hook, rel, step_masks  # noqa: E402
from oracle import lime_oracle as O  # noqa: E402
from oracle.make_golden import case_inputs  # noqa: E402
from oracle.ref_import import make_config  # noqa: E402

DEV = "cuda"
DISCRIMINATION = 10.0


def nrel(a, b):
    """||a - b|| / ||b|| in fp64."""
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return float((a - b).norm() / b.norm())


def judge(name, got, ref, exact, bar_n, bar_e):
    """got vs the rounding reference: norm-relative < bar_n, per element (0.1 rms floor) < bar_e; and >= 10x closer to
    the reference than to exact fp64.  Returns (norm-relative, per-element, distance to exact)."""
    got = got.detach().double().cpu()
    en, ee, ex = nrel(got, ref), rel(got, ref.detach()), nrel(got, exact)
    print("%s: vs rounding reference %.2e (per element %.2e), vs exact fp64 %.2e" % (name, en, ee, ex))
    assert en < bar_n and ee < bar_e, (name, en, ee)
    assert DISCRIMINATION * en <= ex, (name, en, ex)
    return en, ee, ex


def heads_of(x, n, T, heads, hd):
    """[n * T, heads * hd] -> [n, heads, T, hd]"""
    return x.reshape(n, T, heads, hd).transpose(1, 2)


def rows_of(x):
    """[n, heads, T, hd] -> [n * T, heads * hd]"""
    n, heads, T, hd = x.shape
    return x.transpose(1, 2).reshape(n * T, heads * hd)


def gen(seed):
    return torch.Generator(device="cpu").manual_seed(seed)


def draw_qkv(n, heads, T, hd, kind, seed):
    """fp64 q, k, v [n, heads, T, hd]: "normal" logits of unit spread, "sharp" logits up to +-30 (most weights underflow),
    "flat" q = k = 0 (P = 1 / T, exact in bf16)."""
    g = gen(seed)
    sq = {"normal": 1.0, "sharp": 3.2, "flat": 0.0}[kind]
    q, k = (torch.randn(n, heads, T, hd, generator=g, dtype=torch.float64) * sq for _ in range(2))
    v = torch.randn(n, heads, T, hd, generator=g, dtype=torch.float64)
    return q, k, v


# ---------------------------------------------------------------------------------------------
# mha_tc_kernel (lime_mha_bf16, Stage A): head-padded bf16 q | k | v -> bf16 context
# ---------------------------------------------------------------------------------------------
EVAL_BAR_N, EVAL_BAR_E = 3e-4, 8e-2         # measured worst 1.05e-4, 2.6e-2


@pytest.mark.parametrize("T,heads,hd,kind", [
    (32, 10, 30, "normal"), (128, 10, 30, "normal"), (32, 10, 30, "sharp"), (128, 10, 30, "sharp"),
    (32, 10, 30, "flat"), (128, 10, 30, "flat"),
    # T = 32 runs 4 heads per pass: a single partial pass, one full pass, a partial last pass, three full passes
    (32, 1, 32, "normal"), (32, 4, 32, "normal"), (32, 10, 32, "normal"), (32, 12, 32, "normal"), (128, 12, 32, "normal")])
def test_mha_eval_bf16_parity(lib, T, heads, hd, kind):
    n = 12 if T == 32 else 4
    d, rows = heads * hd, n * T
    q, k, v = (bf(x) for x in draw_qkv(n, heads, T, hd, kind, seed=T + heads + hd))
    w = 3 * heads * 32
    ldq, ldo = w + 64, d + 22                                      # strided rows: ldq > 960 at 10 heads, ldo > d
    hp = torch.full((rows, ldq), float("nan"), dtype=torch.float64)  # columns beyond the heads are never read
    hp[:, :w] = 0.0
    qkv_view = hp[:, :w].view(rows, 3, heads, 32)
    for m, x in enumerate((q, k, v)):
        qkv_view[:, m, :, :hd] = x.transpose(1, 2).reshape(rows, heads, hd)
    qkv16 = hp.to(torch.bfloat16).to(DEV)
    out = torch.full((rows, ldo), 7.0, dtype=torch.bfloat16, device=DEV)
    ops.mha_bf16(qkv16, out, n, T, d, heads)
    out = out.cpu()
    assert float(out[:, d:].float().abs().max()) == 0.0           # the canary in columns d..ldo: K padding of out_proj's operand
    got = out[:, :d].double()
    ref, exact = rows_of(mha_eval_bf16(q, k, v)), rows_of(attention_exact(q, k, v))
    assert torch.isfinite(got).all()
    judge("mha_tc T=%d heads=%d hd=%d %s" % (T, heads, hd, kind), got, ref, exact, EVAL_BAR_N, EVAL_BAR_E)


# ---------------------------------------------------------------------------------------------
# mha_fwd_tc_kernel / mha_bwd_tc_kernel (lime_mha_{fwd,bwd}_bf16, the training step's bf16 mode)
# ---------------------------------------------------------------------------------------------
TRAIN_BAR_N, TRAIN_BAR_E = 2e-4, 1.2e-1     # measured worst 6.6e-5, 4.1e-2


def train_reference(qkv, dctx, n, T, d, heads, keep):
    """(ctx, dqkv) of the rounding reference and of exact fp64 attention, [n * T, d] / [n * T, 3 d]."""
    hd = d // heads
    out = {}
    for name, fn in (("ref", lambda q, k, v: Bf16Attention.apply(q, k, v, keep)),
                     ("exact", lambda q, k, v: attention_exact(q, k, v, keep))):
        x = qkv.detach().double().cpu().requires_grad_()
        q, k, v = (heads_of(x[:, i * d:(i + 1) * d], n, T, heads, hd) for i in range(3))
        o = rows_of(fn(q, k, v))
        o.backward(dctx.double().cpu())
        out[name] = (o.detach(), x.grad)
    return out


def run_train_case(n, T, d, heads, p, seed, scale=1.0, misalign=False, kind="normal"):
    rows = n * T
    g = gen(seed)
    base = torch.empty(rows * 3 * d + 1, device=DEV)
    qkv = (base[1:] if misalign else base[:-1]).view(rows, 3 * d)     # 4-byte but not 8-byte aligned: the scalar prologue
    src = torch.randn(rows, 3 * d, generator=g) * scale
    if kind == "flat":
        src[:, :2 * d] = 0.0
    qkv.copy_(src)
    dctx = torch.randn(rows, d, generator=g).to(DEV)
    ctx = torch.empty(rows, d, device=DEV)
    ops.mha(qkv, ctx, n, T, d, heads, p, seed, bf16=True)
    dqkv = ops.mha_bwd(qkv, dctx, n, T, d, heads, p, seed, bf16=True)
    keep = device_keep(seed, [n, heads, T, T], p).double().cpu() if p > 0 else torch.ones(n, heads, T, T, dtype=torch.float64)
    return ctx, dqkv, train_reference(qkv, dctx, n, T, d, heads, keep)


@pytest.mark.parametrize("T,d,heads,p,misalign,kind", [
    (32, 300, 10, 0.0, False, "normal"), (128, 300, 10, 0.0, False, "normal"),
    (32, 300, 10, 0.25, False, "normal"), (128, 300, 10, 0.25, False, "normal"),
    (32, 300, 10, 0.25, False, "sharp"), (128, 300, 10, 0.0, False, "flat"),
    # hd = 27 (odd) and a base 4 bytes off an 8-byte boundary take the scalar-load prologue
    (32, 270, 10, 0.0, False, "normal"), (128, 270, 10, 0.25, False, "normal"),
    (32, 300, 10, 0.25, True, "normal"), (128, 300, 10, 0.0, True, "normal")])
def test_mha_train_bf16_parity(lib, T, d, heads, p, misalign, kind):
    n = 8 if T == 32 else 3
    scale = {"normal": 1.0, "sharp": 3.2, "flat": 1.0}[kind]
    ctx, dqkv, r = run_train_case(n, T, d, heads, p, seed=7 * T + d + int(100 * p), scale=scale, misalign=misalign, kind=kind)
    tag = "mha_%s T=%d d=%d p=%g%s %s" % ("%s", T, d, p, " misaligned" if misalign else "", kind)
    judge(tag % "fwd_tc", ctx, r["ref"][0], r["exact"][0], TRAIN_BAR_N, TRAIN_BAR_E)
    for i, name in enumerate("qkv"):
        cols = slice(i * d, (i + 1) * d)
        if kind == "flat" and name != "v":                        # q = k = 0: dQ = scale dS K and dK = scale dS^T Q vanish
            assert float(dqkv[:, cols].abs().max()) == 0.0, name
            continue
        judge(tag % ("bwd_tc d" + name), dqkv[:, cols], r["ref"][1][:, cols], r["exact"][1][:, cols], TRAIN_BAR_N, TRAIN_BAR_E)


def test_mha_train_bf16_chunk_boundary(lib):
    """65,537 news at T = 32: two launches, the second with news0 = 65,535.  News 65,533..65,536 straddle the boundary;
    their masks are device_keep's at the GLOBAL news index, so a news0 that does not reach the mask index fails here."""
    n, T, d, heads, p, seed = 65537, 32, 300, 10, 0.25, 77
    lo = n - 4
    keep = device_keep(seed, [n * heads * T, T], p)[lo * heads * T:].double().cpu().view(4, heads, T, T)
    torch.cuda.empty_cache()                                # the mask of every news is 2.7 GB; only the last four are kept
    g = torch.Generator(device=DEV).manual_seed(seed)
    qkv = torch.randn(n * T, 3 * d, device=DEV, generator=g)
    dctx = torch.randn(n * T, d, device=DEV, generator=g)
    ctx = torch.empty(n * T, d, device=DEV)
    ops.mha(qkv, ctx, n, T, d, heads, p, seed, bf16=True)
    dqkv = ops.mha_bwd(qkv, dctx, n, T, d, heads, p, seed, bf16=True)
    sl = slice(lo * T, n * T)
    ctx, dqkv, qkv, dctx = ctx[sl].cpu(), dqkv[sl].cpu(), qkv[sl].cpu(), dctx[sl].cpu()
    torch.cuda.empty_cache()
    r = train_reference(qkv, dctx, 4, T, d, heads, keep)
    judge("mha_fwd_tc chunk boundary", ctx, r["ref"][0], r["exact"][0], TRAIN_BAR_N, TRAIN_BAR_E)
    judge("mha_bwd_tc chunk boundary", dqkv, r["ref"][1], r["exact"][1], TRAIN_BAR_N, TRAIN_BAR_E)


# ---------------------------------------------------------------------------------------------
# Stage A bf16 cache build: NewsEncoderEngine.encode_content with bf16 = True
# ---------------------------------------------------------------------------------------------
CONTENT_BAR_N, CONTENT_BAR_E = 2e-4, 1.5e-2  # measured worst 6.0e-5, 4.4e-3


def _stage_a_model(case, golden_dir):
    if case == "small_bs8":
        spec, cfg, news, _ = case_inputs(case)
        n0 = np.load("%s/%s.npz" % (golden_dir, case))["content"].shape[0]
        seed = spec["weights_seed"]
    else:
        cfg = make_config(vocabulary_size=5000, batch_size=32)
        news = synth.make_news_table(600, vocabulary_size=5000, seed=31)
        n0, seed = news.news_num, 7
    cfg.word_embedding_init = "skip"
    model = L.Model(cfg)
    model.initialize()
    synth.synthetic_parameters(model, seed)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    return cfg, news, n0, sd, model.to(DEV).eval()


@pytest.mark.parametrize("case", ["small_bs8", "synth600"])
def test_stage_a_bf16_content_parity(lib, golden_dir, case):
    cfg, news, n0, sd, model = _stage_a_model(case, golden_dir)
    eng = model.news_encoder.engine
    eng.bf16 = True
    dev = lambda a: torch.as_tensor(np.ascontiguousarray(a[:n0], np.int32)).to(DEV)
    with torch.no_grad():
        got = eng.encode_content(dev(news.title_text), dev(news.body_text), dev(news.category), dev(news.subCategory))
        # the in_proj output's head-pad columns are exact zeros (mha_tc_kernel reads all 32 columns of a head): the pad
        # rows of the head-padded weight and the pad entries of its bias are zero, and so is what the GEMM makes of them
        P = eng.prepare()
        hd = 300 // cfg.head_num
        for name in ("title", "body"):
            assert float(P[name]["in_w16"].view(3, cfg.head_num, 32, -1)[:, :, hd:].float().abs().max()) == 0.0, name
            assert float(P[name]["in_b_hp"].view(3, cfg.head_num, 32)[:, :, hd:].abs().max()) == 0.0, name
        E = model.news_encoder.base_news_encoder.word_embedding.weight.detach()
        for name, T, ids in (("title", 32, news.title_text), ("body", 128, news.body_text)):
            rows = n0 * T
            x0 = torch.empty(rows, 300, device=DEV)
            x0b = torch.empty(rows, P[name]["in_w16"].shape[1], dtype=torch.bfloat16, device=DEV)
            ops.embed_pe_bf16(E, dev(ids).reshape(-1), T, P[name + "_pe"], x0, x0b)
            qkv = ops.linear_tma(x0b, P[name]["in_w16"], P[name]["in_b_hp"]).view(rows, 3, cfg.head_num, 32)
            assert float(qkv[..., hd:].float().abs().max()) == 0.0, name
    host = lambda a: torch.as_tensor(np.asarray(a[:n0])).long()
    args = (host(news.title_text), host(news.body_text), host(news.category), host(news.subCategory))
    sd64 = {k: v.double() if v.dtype.is_floating_point else v for k, v in sd.items()}
    ref = crown_content_bf16(sd64, *args, cfg)
    with torch.no_grad():
        exact = torch.cat([O.crown_content(sd64, *(a[lo:lo + 64] for a in args), cfg, torch.float64)
                           for lo in range(0, n0, 64)])
    judge("stage A bf16 content %s (%d news)" % (case, n0), got, ref, exact, CONTENT_BAR_N, CONTENT_BAR_E)


# ---------------------------------------------------------------------------------------------
# the bf16 training step: training.encode_news and training.model_forward with A.set_bf16(True)
# ---------------------------------------------------------------------------------------------
# The step chains a dozen bf16 roundings.  Before each one the device's fp32 value and the fp64 reference's differ by the
# error gathered so far (delta), so a fraction ~delta / ulp of the rounded values land one ulp apart, which adds ~sqrt(delta
# ulp) of error: the discrimination against exact fp64 shrinks along the chain and is asserted at its measured size below.
# The same hooked oracle evaluated in fp32 on the host (the same rounding points, fp32 arithmetic as the device's) carries
# that floor too, and bounds the kernel's distance: a rounding point the reference placed wrongly would put the device
# far outside it.
# (norm-relative bar, least distance to exact fp64 over the distance to the rounding reference); for gradients the bar of
# every parameter and the ratio of the whole gradient vector.  Measured on a B200: encode_news vectors 4.2e-4, x7.7;
# its gradients worst 1.45e-2, whole vector 2.4e-3, x4.3; step logits 3.3e-3, x3.1; step gradients worst 1.37e-2, whole vector 2.4e-3, x3.4.
STEP_BARS = {"encode_news": (1.3e-3, 5.0), "encode_news grad": (4.5e-2, 2.0), "step": (1e-2, 2.0), "step grad": (4.5e-2, 2.0)}
# the device's distance over the host fp32 evaluation's (+ 2e-5 of fp32 accumulation): measured worst 1.8
FP32_FACTOR = 5.5


def _sd(model, dtype):
    return {k: v.detach().clone().to(dtype if v.dtype.is_floating_point else v.dtype).requires_grad_(v.dtype.is_floating_point)
            for k, v in model.state_dict().items()}


def judge_output(tag, got, ref, ref32, exact, bar, ratio):
    got = got.detach().double().cpu()
    en, e32, ex = nrel(got, ref), nrel(ref32.detach(), ref), nrel(got, exact)
    print("%s: vs rounding reference %.2e (host fp32 with the same rounding %.2e), vs exact fp64 %.2e (x%.1f)"
          % (tag, en, e32, ex, ex / en))
    assert en < bar and en <= FP32_FACTOR * (e32 + 2e-5), (tag, en, e32)
    assert ex >= ratio * en, (tag, en, ex)


def judge_step_gradients(tag, params, sds, bar, ratio):
    """Every trainable parameter's gradient against the fp64 rounding reference (norm-relative: single elements of the
    transformer weight gradients move by O(1) of their rms under the one-ulp flips, on the device and on the host alike)
    and, as one vector, the same rules as judge_output.  sds: the state dicts of the fp64 rounding reference, its fp32 evaluation and
    exact fp64, whose .grad the oracle filled."""
    ref, r32, exact = sds
    gmax = max(float(exact[k].grad.abs().max()) for k, q in params if q.requires_grad and exact[k].grad is not None)
    vec, worst, checked = ([], [], [], []), ("", 0.0, 0.0), 0
    for name, prm in params:
        if not prm.requires_grad:
            continue
        g_ex = exact[name].grad
        if g_ex is None or float(g_ex.abs().max()) == 0.0:                  # dead parameters
            assert prm.grad is None or float(prm.grad.abs().max()) == 0.0, name
            continue
        if float(g_ex.abs().max()) < 1e-12 * gmax:                        # zero in exact arithmetic (see test_gpu_training.py)
            assert float(prm.grad.abs().max()) < 1e-10 * gmax, (name, float(prm.grad.abs().max()), gmax)
            continue
        g = prm.grad.double().cpu()
        err, err32 = nrel(g, ref[name].grad), nrel(r32[name].grad, ref[name].grad)
        print("  %s %s: %.2e (host fp32 %.2e)" % (tag, name, err, err32))
        assert err < bar and err <= FP32_FACTOR * (err32 + 2e-5), (tag, name, err, err32)
        worst = max(worst, (name, err, err32), key=lambda t: t[1])
        for v, t in zip(vec, (g, ref[name].grad, r32[name].grad.double(), g_ex)):
            v.append(t.reshape(-1))
        checked += 1
    got, want, w32, ex = (torch.cat(v) for v in vec)
    print("%s: %d gradients, worst %s %.2e (host fp32 %.2e)" % ((tag, checked) + worst))
    judge_output(tag + " (all gradients)", got, want, w32, ex, bar, ratio)
    return checked


def test_news_encoder_bf16_parity(lib):
    """The bf16 twin of tests/test_gpu_training.py::test_news_encoder_gradients: 41 news through training.encode_news."""
    cfg = make_config(vocabulary_size=500, batch_size=4, word_embedding_init="skip", dropout_rate=0.0)
    model = L.Model(cfg)
    model.initialize()
    synth.synthetic_parameters(model, 21)
    sds = (_sd(model, torch.float64), _sd(model, torch.float32), _sd(model, torch.float64))
    model = model.to(DEV).train()
    news = synth.make_news_table(40, vocabulary_size=cfg.vocabulary_size, seed=3)
    n = news.news_num
    rng = np.random.default_rng(5)
    fresh = np.exp(rng.uniform(0, 16, n)).astype(np.float32)
    life = np.exp(rng.uniform(6, 13, n)).astype(np.float32)
    R = torch.randn(n, 400, generator=gen(9), dtype=torch.float64)
    t32 = lambda a: torch.as_tensor(np.ascontiguousarray(a, np.int32)).to(DEV)
    A.set_bf16(True)
    try:
        v = training.encode_news(model.news_encoder, t32(news.title_text), t32(news.body_text), t32(news.category),
                                 t32(news.subCategory), torch.as_tensor(fresh).to(DEV), torch.as_tensor(life).to(DEV))
        (v * R.float().to(DEV)).sum().backward()
    finally:
        A.set_bf16(False)
    tl = lambda a: torch.as_tensor(np.asarray(a)).long()
    args = (tl(news.title_text), tl(news.body_text), tl(news.category), tl(news.subCategory), torch.as_tensor(fresh),
            torch.as_tensor(life), cfg)
    out = []
    for sd, dt, hooks in zip(sds, (torch.float64, torch.float32, torch.float64),
                             (dict(mm=train_mm, attn=bf16_attn), dict(mm=train_mm, attn=bf16_attn), {})):
        w = O.lime_news(sd, *args, dt, **hooks)
        (w * R.to(dt)).sum().backward()
        out.append(w.detach())
    bar, ratio = STEP_BARS["encode_news"]
    judge_output("bf16 encode_news vectors", v, *out, bar, ratio)
    params = [(k, q) for k, q in model.named_parameters() if k.startswith("news_encoder.")]
    assert judge_step_gradients("bf16 encode_news", params, sds, *STEP_BARS["encode_news grad"]) >= 40


def test_training_step_bf16_parity(lib):
    """training.model_forward in bf16 mode with dropout 0.2 at every site and a runtime batch B = 14 > H = 10 (user-node
    rows in the GraphSAGE mean), as tests/test_gpu_training_parity.py::test_training_step_with_dropout_and_user_node_rows:
    logits and every trainable parameter's gradient against the oracle with the bf16 hooks and the same masks."""
    H, B, negatives, p = 10, 14, 4, 0.2
    N = 1 + negatives
    cfg = make_config(vocabulary_size=500, batch_size=16, max_history_num=H, word_embedding_init="skip", dropout_rate=p)
    model = L.Model(cfg)
    model.initialize()
    synth.synthetic_parameters(model, 51)
    p_ca = model.user_encoder.candidate_aware_attn.dropout.p
    sds = (_sd(model, torch.float64), _sd(model, torch.float32), _sd(model, torch.float64))
    model = model.to(DEV).train()
    news = synth.make_news_table(60, vocabulary_size=cfg.vocabulary_size, seed=4)
    batch = list(synth.make_train_batch(news, B, max_history=H, negatives=negatives, seed=6))
    batch[11] = batch[11].copy()
    batch[11][0, 4:] = False                                       # a short history
    batch[11][1, :] = False                                        # an empty one
    tb = [torch.as_tensor(x).to(DEV) for x in batch]
    A.set_bf16(True)
    try:
        logits = training.model_forward(model, tb[1], tb[2], tb[3], tb[6], tb[9], tb[10], tb[11], tb[15], tb[16], tb[17],
                                        tb[20], tb[23], tb[24], tb[24] - tb[23], seed=STEP_SEED)
        (-torch.log_softmax(logits, dim=1)[:, 0]).mean().backward()
    finally:
        A.set_bf16(False)
    masks = step_masks(cfg, B, H, N, p, p_ca, batch[3].shape[-1], batch[6].shape[-1])
    drop = oracle_hook(masks, B * H)
    out = []
    for sd, dt, hooks in zip(sds, (torch.float64, torch.float32, torch.float64),
                             (dict(mm=train_mm, attn=bf16_attn), dict(mm=train_mm, attn=bf16_attn), {})):
        w = O.model_forward(sd, batch, cfg, dt, prefix_len=B, drop=drop, **hooks)
        (-torch.log_softmax(w, dim=1)[:, 0]).mean().backward()
        out.append(w.detach())
    bar, ratio = STEP_BARS["step"]
    judge_output("bf16 training step logits", logits, *out, bar, ratio)
    assert judge_step_gradients("bf16 training step", list(model.named_parameters()), sds, *STEP_BARS["step grad"]) >= 60
