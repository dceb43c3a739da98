"""The bf16 modes' rounding contract restated in fp64: every value is exact except where a kernel rounds to bf16, and
there it is rounded as the kernel rounds it (``bf``: round to nearest even, of the fp32 value the kernel holds).  What is
left between a kernel and these references is fp32 accumulation plus rare one-ulp flips of a rounded value, so the bf16
paths can be held to bars one to three orders of magnitude below bf16 rounding itself.

Rounding points, as the kernels place them (csrc/news_kernels.cu, csrc/gemm_tma.cu, autograd.py, engine.py):

- mha_tc_kernel (eval, lime_mha_bf16): bf16 q | k | v; S = Q K^T; P~ = exp((S - rowmax) / sqrt(hd)) unnormalised;
  l = sum P~ (unrounded); ctx = bf(bf(P~) V / l).
- mha_fwd_tc_kernel (training forward): q, k, v rounded in the prologue; l = sum P~ before the dropout mask M;
  O = bf(P~ M) V / l in fp32.
- mha_bwd_tc_kernel (training backward): q, k, v, dO rounded; P = P~ / l in fp32; dP = M (bf(dO) bf(V)^T);
  rowdot = sum P dP of the unrounded P; dS = P (dP - rowdot); dQ = scale bf(dS) K, dK = scale bf(dS)^T Q,
  dV = bf(P M)^T dO.
- bf16 Linear (autograd.Linear in bf16 mode): y = act(bf(x) bf(w)^T + b) + r; dz = act'(y) dy; dx = bf(dz) bf(w),
  dw = bf(dz)^T bf(x), db = sum dz unrounded.
- Stage A bf16 branch (engine._branch_bf16): the four transformer products as bf16 Linear forwards, the in_proj output
  (q | k | v) rounded, the attention context rounded, the residual stream and LayerNorms in fp32; the small layers
  after the branches run as fp32x3 passes (2^-21 per product) and are exact here.
"""
from __future__ import annotations

import math

import torch

from oracle import lime_oracle as O


def bf(x):
    """Round to nearest even bf16 of the fp32 value, returned in x's dtype (fp64 here)."""
    return x.float().to(torch.bfloat16).to(x.dtype)


def _scores(q, k):
    s = q @ k.transpose(-1, -2)
    return torch.exp((s - s.amax(dim=-1, keepdim=True)) / math.sqrt(q.shape[-1]))


def attention_exact(q, k, v, keep=None):
    """softmax(q k^T / sqrt(hd)) (* keep) @ v in the inputs' precision, no rounding: [..., T, hd]."""
    w = torch.softmax((q @ k.transpose(-1, -2)) / math.sqrt(q.shape[-1]), dim=-1)
    return (w if keep is None else w * keep) @ v


def mha_eval_bf16(q, k, v):
    """mha_tc_kernel: [..., T, hd] head slices -> the bf16 context (as fp64)."""
    q, k, v = bf(q), bf(k), bf(v)
    p = _scores(q, k)
    return bf((bf(p) @ v) / p.sum(dim=-1, keepdim=True))


class Bf16Attention(torch.autograd.Function):
    """mha_fwd_tc_kernel forward and mha_bwd_tc_kernel backward: q, k, v [..., T, hd], keep [..., T, T] (the dropout
    mask keep / (1 - p), ones without dropout) -> O [..., T, hd]; gradients flow to q, k, v only."""

    @staticmethod
    def forward(ctx, q, k, v, keep):
        q, k, v = bf(q), bf(k), bf(v)
        p = _scores(q, k)
        l = p.sum(dim=-1, keepdim=True)                    # before the mask
        ctx.save_for_backward(q, k, v, keep, p / l)
        return (bf(p * keep) @ v) / l

    @staticmethod
    def backward(ctx, dout):
        q, k, v, keep, p = ctx.saved_tensors
        scale = 1.0 / math.sqrt(q.shape[-1])
        do = bf(dout)
        dp = keep * (do @ v.transpose(-1, -2))
        ds = p * (dp - (p * dp).sum(dim=-1, keepdim=True))  # rowdot of the unrounded P
        dsb = bf(ds)
        return scale * dsb @ k, scale * dsb.transpose(-1, -2) @ q, bf(p * keep).transpose(-1, -2) @ do, None


class Bf16Linear(torch.autograd.Function):
    """bf(x) @ bf(w).T and the bf16-mode backward: dx = bf(dz) bf(w), dw = bf(dz)^T bf(x) (bias and activation are
    applied outside, so their gradients stay unrounded as in autograd.Linear)."""

    @staticmethod
    def forward(ctx, x, w):
        xb, wb = bf(x), bf(w)
        ctx.save_for_backward(xb, wb)
        return xb @ wb.t()

    @staticmethod
    def backward(ctx, dz):
        xb, wb = ctx.saved_tensors
        dzb = bf(dz)
        dw = dzb.reshape(-1, wb.shape[0]).t() @ xb.reshape(-1, wb.shape[1])
        return dzb @ wb, dw


FRESHNESS_DENSE = O.NEWS + "freshness_encoder.dense"


def train_mm(prefix, x, w):
    """The oracle's ``mm`` hook for the bf16 training step: every product as a bf16 Linear.  The freshness dense layer
    runs once per bucket pair on the device (training.encode_news: a [nb * nb] table, then a gather), so its dz is summed
    over the news of a bucket pair before it is rounded: the same here, by evaluating the layer on the distinct rows."""
    if prefix != FRESHNESS_DENSE:
        return Bf16Linear.apply(x, w)
    u, inv = torch.unique(x.detach(), dim=0, return_inverse=True)
    rows = inv.new_empty(u.shape[0]).scatter_(0, inv, torch.arange(x.shape[0]))    # one news per distinct row
    return Bf16Linear.apply(x[rows], w)[inv]


def bf16_attn(q, k, v, drop_attn):
    """The oracle's ``attn`` hook of the bf16 attention cores: the training forward under the "attn" dropout site, and
    without dropout the Stage A core up to the context's rounding, which the next product (out_proj) repeats."""
    keep = drop_attn(torch.ones(q.shape[:-1] + (k.shape[-2],), dtype=q.dtype))
    return Bf16Attention.apply(q, k, v, keep)


def stage_a_mm(prefix, x, w):
    """The ``mm`` hook of the Stage A bf16 mode: bf16 products in the transformer branches only."""
    return Bf16Linear.apply(x, w) if "_transformer." in prefix else x @ w.t()


def crown_content_bf16(sd, title_text, body_text, category, subCategory, cfg, chunk=64):
    """fp64 restatement of NewsEncoderEngine.encode_content in bf16 mode -> [n, 900], ``chunk`` news at a time."""
    out = []
    with torch.no_grad():
        for lo in range(0, title_text.shape[0], chunk):
            s = slice(lo, lo + chunk)
            out.append(O.crown_content(sd, title_text[s], body_text[s], category[s], subCategory[s], cfg, torch.float64,
                                       mm=stage_a_mm, attn=bf16_attn))
    return torch.cat(out)
