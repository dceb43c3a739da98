"""Parity of the training path with dropout on: every non-GEMM training kernel (csrc/train_user.cu and the news-side
intent-pool / content-fuse backward) against fp64 torch autograd of the same formulas, at the shapes and edges where
such kernels go wrong, and one whole training step with every dropout site live and user-node rows in the GraphSAGE
mean (runtime batch > max_history_num) against the fp64 oracle run under the same masks.

Every mask is read from the library's own generator (``device_keep``): the kernels compare a 32-bit draw rounded to
fp32 with fp32 p, which a host restatement of the hash would have to reproduce bit for bit."""
import math
import types

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import lime_cikm25_b200 as L  # noqa: E402
from lime_cikm25_b200 import _lib, ops, synth, training  # noqa: E402
from lime_cikm25_b200 import autograd as A  # noqa: E402
from oracle import lime_oracle as O  # noqa: E402
from oracle.ref_import import make_config  # noqa: E402

DEV = "cuda"
D = 400          # user-side vector width (LIME output)
HEADS = 10       # heads of the candidate-aware attention (layers.py:22)
TOL = 5e-5


def rms(b):
    return float(np.sqrt(np.mean(np.asarray(b, np.float64) ** 2)))


def rel(a, b, floor=0.0):
    """Max relative error, each element against max(|b|, 0.1 rms(b)) (the measure of tests/test_gpu_training.py), or
    against ``floor`` where that is larger."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    floor = max(0.1 * rms(b), floor) + 1e-30
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), floor)))


def check(pairs, tol=TOL, floors=None, fp32=None):
    """pairs: {name: (device tensor, fp64 reference)} -> worst error; fails on the first one above tol.
    floors: {name: absolute floor of the error measure} for outputs whose exact value may vanish.
    fp32: {name: the reference's formulas evaluated by torch in fp32}: where fp32 itself is ill-conditioned (the softmax
    and sigmoid backward a (g - sum a g), g (1 - g) lose digits when one weight nears 1) an error within 4x of torch-fp32's
    is accepted too, as tests/test_gpu_training.py::test_news_encoder_gradients accepts it."""
    worst = 0.0
    for name, (got, want) in pairs.items():
        assert tuple(got.shape) == tuple(want.shape), (name, tuple(got.shape), tuple(want.shape))
        floor = (floors or {}).get(name, 0.0)
        err = rel(got.detach().cpu(), want.detach(), floor)
        if err >= tol and fp32 is not None:
            err32 = rel(fp32[name].detach(), want.detach(), floor)
            assert err < 4 * err32, (name, err, err32)
        else:
            assert err < tol, (name, err)
        worst = max(worst, err)
    return worst


def gen(seed):
    return torch.Generator(device="cpu").manual_seed(seed)


def randn(*shape, seed=0, scale=1.0):
    return (torch.randn(*shape, generator=gen(seed)) * scale).to(DEV)


def f64(t):
    return t.detach().double().cpu().requires_grad_()


def device_keep(seed, shape, p):
    """keep / (1 - p) of the stateless dropout at flat index i of ``shape`` under ``seed``: lime_dropout of a ones
    matrix, whose element (r, c) is index r * cols + c.  The only source of masks in this file."""
    rows = math.prod(shape[:-1])
    return ops.dropout(torch.ones(rows, shape[-1], device=DEV), p, seed).view(*shape)


def launches(lib):
    return int(lib.lime_launch_count())


def test_device_keep_is_inverted_dropout(lib):
    k = device_keep(5, [64, 10, 33], 0.2).cpu()
    vals = k.unique()
    assert len(vals) == 2 and float(vals[0]) == 0.0 and float(vals[1]) == 1.25          # 1.0f / (1.0f - 0.2f)
    assert abs(float((k > 0).double().mean()) - 0.8) < 0.01
    assert not torch.equal(k, device_keep(6, [64, 10, 33], 0.2).cpu())
    assert torch.equal(device_keep(5, [640, 33], 0.2).cpu().view(64, 10, 33), k)     # a function of the flat index only


# ---------------------------------------------------------------------------------------------
# candidate-aware attention weights (layers.py:66-81)
# ---------------------------------------------------------------------------------------------
def ca_reference(Q, K, mask, B, N, H, keep):
    """fp64: Q [B*N, 400], K [B*H, 400], mask [B, H] -> a [B*H]; keep [B, 10, N, H] on the post-softmax weights."""
    hd = D // HEADS
    Qh = Q.view(B, N, HEADS, hd).transpose(1, 2)
    Kh = K.view(B, H, HEADS, hd).transpose(1, 2)
    s = (Qh @ Kh.transpose(-1, -2)) / D ** 0.5
    s = s.masked_fill(mask.view(B, 1, 1, H) == 0, -1e9)
    w = torch.softmax(s, dim=-1)
    if keep is not None:
        w = w * keep
    qw = torch.softmax(Q.view(B, N, D).norm(dim=-1), dim=1)
    agg = (w.sum(dim=1) * qw.unsqueeze(-1)).sum(dim=1)
    return torch.softmax(agg, dim=-1).reshape(-1)


def ca_masks(B, H, seed):
    """Random history masks, then every slot masked, a single unmasked slot, only the last slot unmasked."""
    g = gen(seed)
    rand = (torch.rand(B, H, generator=g) < 0.7).to(torch.uint8)
    one = torch.zeros(B, H, dtype=torch.uint8)
    one[torch.arange(B), torch.randint(0, H, (B,), generator=g)] = 1
    last = torch.zeros(B, H, dtype=torch.uint8)
    last[:, -1] = 1
    return {"random": rand, "all_masked": torch.zeros(B, H, dtype=torch.uint8), "single": one, "last": last}


CA_SHAPES = [(1, 1, 1), (3, 5, 50), (2, 1, 64), (5, 5, 33), (2, 64, 8), (3, 41, 50)]


@pytest.mark.parametrize("p", [0.0, 0.2])
@pytest.mark.parametrize("B,N,H", CA_SHAPES)
def test_ca_attention_forward_backward(lib, B, N, H, p):
    seed = 1000 + B * 7 + N * 13 + H
    Qp, Kp = randn(B * N, D, seed=seed, scale=2.0), randn(B * H, D, seed=seed + 1, scale=2.0)
    da = randn(B * H, seed=seed + 2)
    keep = device_keep(seed, [B, HEADS, N, H], p).double().cpu() if p > 0 else None
    worst, floors = 0.0, None
    for kind, mask in ca_masks(B, H, seed).items():
        m = mask.to(DEV)
        a = ops.ca_attention_fwd(Qp, Kp, m, B, N, H, p, seed)
        dQ, dK = ops.ca_attention_bwd(Qp, Kp, m, B, N, H, da, p, seed)
        ref = {}
        for dt in (torch.float64, torch.float32):
            Qr, Kr = (t.detach().cpu().to(dt).requires_grad_() for t in (Qp, Kp))
            ar = ca_reference(Qr, Kr, mask, B, N, H, None if keep is None else keep.to(dt))
            ar.backward(da.cpu().to(dt))
            ref[dt] = (ar, Qr.grad, Kr.grad)
        want, dQ64, dK64 = ref[torch.float64]
        pairs = {"a": (a, want), "dQ": (dQ, dQ64), "dK": (dK, dK64)}
        # With one slot (or none) unmasked the exact dQ is 0 for p = 0 (and for N = 1), or a small difference of
        # equal-sized terms: errors are measured against each output's size at the random mask of the same inputs.
        floors = floors or {k: 0.1 * rms(w.detach()) for k, (_, w) in pairs.items()}
        try:
            worst = max(worst, check(pairs, floors=floors, fp32=dict(zip(("a", "dQ", "dK"), ref[torch.float32]))))
        except AssertionError as e:
            raise AssertionError((kind,) + e.args) from None
        if kind == "all_masked":                # no gradient reaches the logits of masked slots
            assert float(dK.abs().max()) == 0.0
    print("ca_attention B=%d N=%d H=%d p=%g: worst %.2e" % (B, N, H, p, worst))


def test_ca_attention_forward_and_backward_admit_the_same_shapes(lib):
    """Both directions share one shared-memory limit: at H = 50, N = 41 runs forward and backward, N = 42 is rejected by
    both (its forward used to run and its backward to fail)."""
    H, B = 50, 2
    for N, ok in ((41, True), (42, False)):
        Qp, Kp = randn(B * N, D, seed=N), randn(B * H, D, seed=N + 1)
        m = torch.ones(B, H, dtype=torch.uint8, device=DEV)
        da = randn(B * H, seed=3)
        for call in (lambda: ops.ca_attention_fwd(Qp, Kp, m, B, N, H, 0.2, 9),
                     lambda: ops.ca_attention_bwd(Qp, Kp, m, B, N, H, da, 0.2, 9)):
            n0 = launches(lib)
            if ok:
                call()
                torch.cuda.synchronize()
                assert launches(lib) == n0 + 1
            else:
                with pytest.raises(_lib.LimeError):
                    call()
                assert launches(lib) == n0


# ---------------------------------------------------------------------------------------------
# row scale, gate mix (layers.py:84-88)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rows", [1, 7, 8, 9, 2500])
def test_row_scale_and_gate_mix(lib, rows):
    v, a = randn(rows, D, seed=rows), randn(rows, seed=rows + 1)
    g = randn(rows, D, seed=rows + 2)
    out = ops.row_scale_fwd(v, a)
    dv, da = ops.row_scale_bwd(v, a, g)
    v64, a64 = f64(v), f64(a)
    want = a64.unsqueeze(1) * v64
    want.backward(g.double().cpu())
    worst = check({"wc": (out, want), "dv": (dv, v64.grad), "da": (da, a64.grad)})
    # z up to +-30: the sigmoid saturates to exactly 0 / 1 in fp32
    z = ((torch.rand(rows, D, generator=gen(rows + 3)) * 2 - 1) * 30).to(DEV)
    z.view(-1)[:2] = torch.tensor([30.0, -30.0])
    wc, x = randn(rows, D, seed=rows + 4), randn(rows, D, seed=rows + 5)
    o = ops.gate_mix_fwd(z, wc, x)
    dz, dwc, dx = ops.gate_mix_bwd(z, wc, x, g)
    ref = {}
    for dt in (torch.float64, torch.float32):
        zr, wr, xr = (t.detach().cpu().to(dt).requires_grad_() for t in (z, wc, x))
        s = torch.sigmoid(zr)
        o_r = s * wr + (1 - s) * xr
        o_r.backward(g.cpu().to(dt))
        ref[dt] = {"o": o_r, "dz": zr.grad, "dwc": wr.grad, "dv": xr.grad}
    got = {"o": o, "dz": dz, "dwc": dwc, "dv": dx}
    worst = max(worst, check({k: (got[k], ref[torch.float64][k]) for k in got}, fp32=ref[torch.float32]))
    print("row_scale / gate_mix rows=%d: worst %.2e" % (rows, worst))


# ---------------------------------------------------------------------------------------------
# GraphSAGE mean over [x_b ; user-node rows] (userEncoders.py:91-98,121,153)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("un_rows", [1, 32, 64])
@pytest.mark.parametrize("B", [1, 3, 64])
def test_sage_mean_forward_backward(lib, B, un_rows):
    """B = 64 at H = 50 runs the grid-stride loop of the backward (B*H*400 elements > 4096 blocks of 256)."""
    H = 50
    x, un = randn(B * H, D, seed=B), randn(un_rows, D, seed=un_rows + 100)
    dm = randn(B, D, seed=B + 200)
    worst = 0.0
    for P in sorted({1, H - 1, H, H + 1, H + un_rows}):
        m = ops.sage_mean_fwd(x, un, B, H, P)
        dx, dun = ops.sage_mean_bwd(dm, B, H, P, un_rows)
        x64, un64 = f64(x), f64(un)
        nodes = torch.cat([x64.view(B, H, D), un64.unsqueeze(0).expand(B, -1, -1)], dim=1)
        want = nodes[:, :P].mean(dim=1)
        want.backward(dm.double().cpu())
        worst = max(worst, check({"m": (m, want), "dx": (dx, x64.grad), "dun": (dun, un64.grad)}))
        pu = max(P - H, 0)                       # user-node rows in the mean
        if pu < un_rows:
            assert float(dun[pu:].abs().max()) == 0.0, P
        if pu > 0:
            assert float(dun[:pu].abs().min()) > 0.0, P
        if P < H:
            assert float(dx.view(B, H, D)[:, P:].abs().max()) == 0.0, P
    print("sage_mean B=%d un_rows=%d: worst %.2e" % (B, un_rows, worst))


@pytest.mark.parametrize("B,H", [(4, 50), (3, 33), (64, 50), (14, 10)])
def test_add_row_bcast_and_sum_over_h(lib, B, H):
    """g[b,h] = r[b,h] + l[b] and its backward; 99 and 140 rows are not multiples of 256."""
    r, l = randn(B * H, D, seed=B), randn(B, D, seed=H)
    g = ops.add_row_bcast(r, l, H)
    assert torch.equal(g, (r.view(B, H, D) + l.unsqueeze(1)).view(B * H, D))     # one fp32 add: exact
    dg = randn(B * H, D, seed=B + H)
    dl = ops.sum_over_h(dg, B, H)
    print("sum_over_h B=%d H=%d: %.2e" % (B, H, check({"dl": (dl, dg.double().cpu().view(B, H, D).sum(1))})))


# ---------------------------------------------------------------------------------------------
# candidate-query pooling (userEncoders.py:158-171)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,H", [(1, 1), (5, 50), (41, 50), (64, 64), (200, 64)])
def test_pool_forward_backward(lib, N, H):
    """(200, 64) needs 51,200 B of shared memory: the opt-in path above 48,000 B."""
    B = 3
    Kg, q, g = randn(B * H, D, seed=N), randn(B * N, D, seed=N + 1, scale=2.0), randn(B * H, D, seed=N + 2)
    du = randn(B * N, D, seed=N + 3)
    u, alpha = ops.pool_fwd(Kg, q, g, B, N, H)
    dKg, dq, dg = ops.pool_bwd(Kg, q, g, alpha, du, B, N, H)
    K64, q64, g64 = f64(Kg), f64(q), f64(g)
    al = torch.softmax(q64.view(B, N, D) @ K64.view(B, H, D).transpose(1, 2) / D ** 0.5, dim=-1)
    want = (al @ g64.view(B, H, D)).reshape(B * N, D)
    want.backward(du.double().cpu())
    worst = check({"u": (u, want), "alpha": (alpha, al.reshape(B * N, H)), "dKg": (dKg, K64.grad), "dq": (dq, q64.grad),
                   "dg": (dg, g64.grad)})
    print("pool N=%d H=%d: worst %.2e" % (N, H, worst))


# ---------------------------------------------------------------------------------------------
# click score with remaining-lifetime weighting (util.py:23-49)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("use_w,use_pen", [(True, True), (True, False), (False, True), (False, False)])
def test_click_score_forward_backward(lib, use_w, use_pen):
    rows = 1003
    u, c = randn(rows, D, seed=1, scale=0.1), randn(rows, D, seed=2, scale=0.1)
    rem = torch.randn(rows, generator=gen(3)) * 20
    rem[:12] = torch.tensor([-1e6, 1e6, 0.0, -0.0, -0.5, 0.5, -0.999, 0.25, -1.0, 1.0, -3.0, 3.0])
    rem[12:40] = rem[12:40] * 1e-3
    cfg = types.SimpleNamespace(use_remaining_lifetime_weighting=use_w, use_expired_penalty=use_pen,
                                sigmoid_scaling_alpha=0.3, penalty_scaling_beta=0.3)
    s, w = ops.click_score_fwd(u, c, rem.to(DEV), 0.3, 0.3, use_w, use_pen)
    ds = randn(rows, seed=4)
    du, dc = ops.click_score_bwd(u, c, w, ds)
    w64 = O.lifetime_weight(rem.double(), cfg)
    u64, c64 = f64(u), f64(c)
    want = (u64 * c64).sum(-1) * w64
    want.backward(ds.double().cpu())
    worst = check({"w": (w, w64), "s": (s, want), "du": (du, u64.grad), "dc": (dc, c64.grad)})
    assert torch.equal(w.cpu() == 0, w64 == 0)
    print("click_score w=%d pen=%d: worst %.2e" % (use_w, use_pen, worst))


# ---------------------------------------------------------------------------------------------
# news side: intent pooling backward (layers.py:285-300), content fuse backward (newsEncoders.py:222-224,297-300,367-371)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 33, 1000])
def test_intent_pool_backward(lib, n):
    k = 3
    pre, e = randn(n * k, D, seed=n), randn(n * k, D, seed=n + 1).relu()
    w2, dout = randn(D, seed=n + 2, scale=0.07), randn(n, D, seed=n + 3)
    out = ops.intent_pool(pre, e.view(n, k * D), w2, torch.empty(n, D, device=DEV), n, k, D)
    dpre, de, dw2 = ops.intent_pool_bwd(pre, e, w2, dout, n, k, D)
    pre64, e64, w64 = f64(pre), f64(e), f64(w2)
    alpha = torch.softmax(torch.tanh(pre64.view(n, k, D)) @ w64, dim=1)
    want = (alpha.unsqueeze(-1) * e64.view(n, k, D)).sum(1)
    want.backward(dout.double().cpu())
    worst = check({"out": (out, want), "dpre": (dpre, pre64.grad), "de": (de, e64.grad), "dw2": (dw2, w64.grad)})
    print("intent_pool_bwd n=%d: worst %.2e" % (n, worst))


@pytest.mark.parametrize("p", [0.0, 0.2])
def test_content_fuse_backward(lib, p):
    """Through autograd.ContentFuse: [title | sim * body | dropout(cat_emb[c]) | dropout(sub_emb[s])] and its backward,
    including body rows that are positive and negative multiples of their title row (cos = +-1)."""
    n, seed = 37, 4242
    title, body = randn(n, D, seed=1).relu(), randn(n, D, seed=2).relu()
    body[3] = 2.5 * title[3]
    body[5] = -0.75 * title[5]
    title.requires_grad_()
    body.requires_grad_()
    ct = (torch.rand(18, 50, generator=gen(3)) * 0.2 - 0.1).to(DEV).requires_grad_()
    st = (torch.rand(270, 50, generator=gen(4)) * 0.2 - 0.1).to(DEV)
    cat = torch.randint(0, 18, (n,), generator=gen(5)).to(torch.int32)
    sub = torch.randint(0, 270, (n,), generator=gen(6)).to(torch.int32)
    out = A.ContentFuse.apply(title, body, ct, st, cat.to(DEV), sub.to(DEV), p, seed)
    g = randn(n, 2 * D + 100, seed=7)
    out.backward(g)
    t64, b64, ct64 = f64(title), f64(body), f64(ct)
    sim = ((torch.nn.functional.cosine_similarity(t64, b64, dim=1) + 1) / 2).unsqueeze(1)
    ce, se = ct64[cat.long()], st.double().cpu()[sub.long()]
    if p > 0:
        kc, ks = device_keep(seed, [n, 50], p).double().cpu(), device_keep(seed + 1, [n, 50], p).double().cpu()
        assert torch.equal(out[:, 2 * D:2 * D + 50].detach().cpu() == 0, kc == 0)
        assert torch.equal(out[:, 2 * D + 50:].detach().cpu() == 0, ks == 0)
        ce, se = ce * kc, se * ks
    want = torch.cat([t64, sim * b64, ce, se], dim=1)
    want.backward(g.double().cpu())
    worst = check({"out": (out, want), "dtitle": (title.grad, t64.grad), "dbody": (body.grad, b64.grad),
                   "dcat_table": (ct.grad, ct64.grad)})
    print("content_fuse p=%g: worst %.2e" % (p, worst))


# ---------------------------------------------------------------------------------------------
# argument rejection: LimeError, nothing launched
# ---------------------------------------------------------------------------------------------
def test_rejected_arguments_launch_nothing(lib):
    f = lambda *s: torch.zeros(*s, device=DEV)
    mask = lambda B, H: torch.ones(B, H, dtype=torch.uint8, device=DEV)
    calls = []
    for N, H in ((65, 8), (8, 65), (64, 64), (42, 50)):                      # > 64, or over the shared-memory limit
        calls.append(lambda N=N, H=H: ops.ca_attention_fwd(f(2 * N, D), f(2 * H, D), mask(2, H), 2, N, H))
        calls.append(lambda N=N, H=H: ops.ca_attention_bwd(f(2 * N, D), f(2 * H, D), mask(2, H), 2, N, H, f(2 * H)))
    for P in (0, 50 + 16 + 1):                                                # H = 50, 16 user-node rows
        calls.append(lambda P=P: ops.sage_mean_fwd(f(100, D), f(16, D), 2, 50, P))
        calls.append(lambda P=P: ops.sage_mean_bwd(f(2, D), 2, 50, P, 16))
    N, H = 626, 64                                                            # 160,256 B of logits
    calls.append(lambda: ops.pool_fwd(f(H, D), f(N, D), f(H, D), 1, N, H))
    calls.append(lambda: ops.pool_bwd(f(H, D), f(N, D), f(H, D), f(N, H), f(N, D), 1, N, H))
    torch.cuda.synchronize()
    for i, call in enumerate(calls):
        n0 = launches(lib)
        with pytest.raises(_lib.LimeError):
            call()
        assert launches(lib) == n0, i


# ---------------------------------------------------------------------------------------------
# one training step, dropout on, runtime batch B = 14 > H = 10: user-node rows 0-3 enter the GraphSAGE mean
# ---------------------------------------------------------------------------------------------
STEP_SEED = 5000


def step_masks(cfg, B, H, N, p, p_ca, T, Lb):
    """Every dropout site of training.model_forward(seed=STEP_SEED), in the device's flat layouts, as fp64 CPU tensors.
    News rows are the B*H history news, then the B*N candidates (the oracle's "hist." / "cand." prefixes)."""
    s, n = STEP_SEED, B * H + B * N
    d, ff, heads = cfg.word_embedding_dim, cfg.feedforward_dim, cfg.head_num
    keep = lambda seed, shape, q: device_keep(seed, shape, q).double().cpu() if q > 0 else None
    m = {}
    for br, base, t in (("title", 11, T), ("body", 23, Lb)):
        for site, off, shape in (("embed", 0, [n, t, d]), ("pe", 1, [n, t, d]), ("attn", 2, [n, heads, t, t]),
                                 ("out_proj", 3, [n, t, d]), ("ffn", 4, [n, t, ff]), ("linear2", 5, [n, t, d])):
            m[br + "." + site] = keep(s + base + off, shape, p)
    m["cat"] = keep(s + 37, [n, cfg.category_embedding_dim], p)
    m["sub"] = keep(s + 38, [n, cfg.subCategory_embedding_dim], p)
    m["user_node"] = keep(s + 51, [cfg.batch_size, D], p)
    m["ca_attn"] = keep(s + 61, [B, HEADS, N, H], p_ca)
    return m


def oracle_hook(masks, n_hist):
    def drop(site, x):
        part, name = site.split(".", 1) if site.startswith(("hist.", "cand.")) else (None, site)
        k = masks[name]
        if k is None:
            return x
        k = k[:n_hist] if part == "hist" else k[n_hist:] if part == "cand" else k
        assert tuple(k.shape) == tuple(x.shape), (site, tuple(k.shape), tuple(x.shape))
        return x * k.to(x.dtype)
    return drop


@pytest.mark.parametrize("p", [0.2, 0.0])
def test_training_step_with_dropout_and_user_node_rows(lib, p):
    """training.model_forward with every dropout site at p (the candidate-aware attention at its fixed 0.2 when p > 0)
    and the reference trainer's loss: logits and EVERY trainable parameter's gradient vs fp64 autograd through the oracle
    under the same masks, torch-fp32 on the oracle as the yardstick (the acceptance rule of
    tests/test_gpu_training.py::test_training_step_gradients).  p = 0 isolates the user-node branch."""
    H, B, negatives = 10, 14, 4
    N = 1 + negatives
    cfg = make_config(vocabulary_size=500, batch_size=16, max_history_num=H, word_embedding_init="skip", dropout_rate=p)
    model = L.Model(cfg)
    model.initialize()
    synth.synthetic_parameters(model, 51)
    p_ca = model.user_encoder.candidate_aware_attn.dropout.p if p > 0 else 0.0
    if p == 0:
        model.user_encoder.candidate_aware_attn.dropout.p = 0.0
    sd = {k: v.detach().clone().double().requires_grad_(v.dtype.is_floating_point) for k, v in model.state_dict().items()}
    model = model.to(DEV).train()
    news = synth.make_news_table(60, vocabulary_size=cfg.vocabulary_size, seed=4)
    batch = list(synth.make_train_batch(news, B, max_history=H, negatives=negatives, seed=6))
    batch[11] = batch[11].copy()
    batch[11][0, 4:] = False                                       # a short history
    batch[11][1, :] = False                                        # an empty one
    tb = [torch.as_tensor(x).to(DEV) for x in batch]
    logits = training.model_forward(model, tb[1], tb[2], tb[3], tb[6], tb[9], tb[10], tb[11], tb[15], tb[16], tb[17],
                                    tb[20], tb[23], tb[24], tb[24] - tb[23], seed=STEP_SEED)
    assert logits.shape == (B, N)
    (-torch.log_softmax(logits, dim=1)[:, 0]).mean().backward()

    masks = step_masks(cfg, B, H, N, p, p_ca, batch[3].shape[-1], batch[6].shape[-1])
    drop = oracle_hook(masks, B * H)
    want = O.model_forward(sd, batch, cfg, torch.float64, prefix_len=B, drop=drop)
    (-torch.log_softmax(want, dim=1)[:, 0]).mean().backward()
    sd32 = {k: t.detach().float().requires_grad_(t.dtype.is_floating_point) for k, t in sd.items()}
    want32 = O.model_forward(sd32, batch, cfg, torch.float32, prefix_len=B, drop=drop)
    (-torch.log_softmax(want32, dim=1)[:, 0]).mean().backward()

    assert np.array_equal(logits.detach().cpu().numpy() == 0, want32.detach().numpy() == 0)
    el, el32 = rel(logits.detach().cpu(), want.detach()), rel(want32.detach(), want.detach())
    assert el < 1e-3 and el < 4 * el32 + 1e-4, (el, el32)
    checked, worst, worst32 = 0, 0.0, 0.0
    gmax = max(float(sd[n].grad.abs().max()) for n, q in model.named_parameters() if q.requires_grad and sd[n].grad is not None)
    for name, prm in model.named_parameters():
        if not prm.requires_grad:
            continue
        g64 = sd[name].grad
        if g64 is None or float(g64.abs().max()) == 0.0:          # dead parameters (ISAB, affine, value_proj, ...)
            assert prm.grad is None or float(prm.grad.abs().max()) == 0.0, name
            continue
        assert prm.grad is not None, name
        if float(g64.abs().max()) < 1e-12 * gmax:                  # zero in exact arithmetic: see test_training_step_gradients
            assert float(prm.grad.abs().max()) < 1e-10 * gmax, (name, float(prm.grad.abs().max()), gmax)
            checked += 1
            continue
        err, err32 = rel(prm.grad.cpu(), g64), rel(sd32[name].grad, g64)
        assert err < 2e-3 or err < 2 * err32 + 2e-4, (name, err, err32)
        worst, worst32 = max(worst, err), max(worst32, err32)
        checked += 1
    assert checked >= 60

    # the runtime batch of 14 takes user-node rows 0..3 into the mean: their gradient is live outside dropped elements
    gun = model.user_encoder.user_node_embedding.grad.cpu()
    live = masks["user_node"][:B - H] != 0 if p > 0 else torch.ones(B - H, D, dtype=torch.bool)
    assert torch.equal(gun[:B - H] != 0, live)
    assert float(gun[B - H:].abs().max()) == 0.0
    print("training step p=%g: %d parameters, logits %.2e (fp32 oracle %.2e), worst gradient %.2e (fp32 oracle %.2e)"
          % (p, checked, el, el32, worst, worst32))
