"""Tensor-level wrappers over the C ABI (include/lime_b200.h).

torch is used for device memory and the current stream only; every computation below is a call
into liblime_b200.so.  Inputs must be CUDA tensors of the stated dtype; nothing is copied or cast
silently except where the docstring says so.
"""
from __future__ import annotations

import ctypes

import torch

from . import _lib
from ._lib import check

ACT_NONE, ACT_RELU, ACT_TANH = 0, 1, 2


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _ptr(t, dtype, name):
    if t is None:
        return None
    if not t.is_cuda:
        raise _lib.LimeError("%s must be a CUDA tensor (no CPU fallback)" % name)
    if t.dtype != dtype:
        raise TypeError("%s must be %s, got %s" % (name, dtype, t.dtype))
    return t.data_ptr()


def _rowmajor(t, name):
    """(pointer-checked tensor, leading dimension) of a 2-D view whose last dim is contiguous."""
    if t.dim() != 2 or t.stride(1) != 1:
        raise ValueError("%s must be 2-D with a contiguous last dimension" % name)
    return t.stride(0)


def bucketize(seconds, num_buckets):
    """FreshnessEncoder.bucketize (newsEncoders.py:53-58): fp32 seconds -> int32 bucket ids."""
    lib = _lib.require_device()
    x = seconds.contiguous()
    out = torch.empty(x.shape, dtype=torch.int32, device=x.device)
    check(lib.lime_bucketize(_ptr(x, torch.float32, "seconds"), x.numel(), int(num_buckets),
                             out.data_ptr(), _stream()), "lime_bucketize")
    return out


def linear(a, w, bias=None, residual=None, act=ACT_NONE, out=None, n=None, k=None, bf16=False):
    """out[m, :n] = act(a[m, :k] @ w[:n, :k].T + bias) + residual.  a, w, residual, out are 2-D views
    with contiguous last dim (arbitrary row stride); k, row strides of a and w multiples of 4."""
    lib = _lib.require_device()
    m = a.shape[0]
    n = w.shape[0] if n is None else n
    k = a.shape[1] if k is None else k
    lda, ldw = _rowmajor(a, "a"), _rowmajor(w, "w")
    if out is None:
        out = torch.empty((m, n), dtype=torch.float32, device=a.device)
    ldc = _rowmajor(out, "out")
    ldr = _rowmajor(residual, "residual") if residual is not None else 0
    fn = lib.lime_linear_bf16 if bf16 else lib.lime_linear
    check(fn(_ptr(a, torch.float32, "a"), lda, _ptr(w, torch.float32, "w"), ldw,
             _ptr(bias, torch.float32, "bias"), _ptr(residual, torch.float32, "residual"), ldr,
             _ptr(out, torch.float32, "out"), ldc, m, n, k, act, _stream()),
          "lime_linear_bf16" if bf16 else "lime_linear")
    return out


def linear_tma(a16, w16, bias=None, residual=None, act=ACT_NONE, out=None, n=None, out_bf16=True, ld_out=None, alpha=1.0):
    """Stage A dense layer on bf16 activations (lime_linear_bf16_tma): a16 [m, kp] bf16, w16 [n, kp] bf16 (kp = the
    contraction length padded to a multiple of 64 with zero columns), bias / residual fp32.  Returns bf16 [m, ld_out]
    (padding columns zero: the next layer's operand) or fp32 [m, n]."""
    lib = _lib.require_device()
    m, kp = a16.shape
    n = w16.shape[0] if n is None else n
    if out is None:
        out = (torch.empty((m, ld_out or n), dtype=torch.bfloat16, device=a16.device) if out_bf16
               else torch.empty((m, n), dtype=torch.float32, device=a16.device))
    ldr = _rowmajor(residual, "residual") if residual is not None else 0
    if a16.dtype != w16.dtype or a16.dtype not in (torch.bfloat16, torch.float16):
        raise TypeError("a16 / w16 must both be bfloat16 or both float16")
    check(lib.lime_linear_bf16_tma(_ptr(a16, a16.dtype, "a16"), _rowmajor(a16, "a16"), _ptr(w16, a16.dtype, "w16"),
                                   _rowmajor(w16, "w16"), _ptr(bias, torch.float32, "bias"),
                                   _ptr(residual, torch.float32, "residual"), ldr, out.data_ptr(), _rowmajor(out, "out"),
                                   1 if out.dtype == torch.bfloat16 else 0, m, n, kp, act, float(alpha),
                                   1 if a16.dtype == torch.float16 else 0, _stream()), "lime_linear_bf16_tma")
    return out


ACT_RES_FIRST = 16


def split16(x, kp=None, scale=1.0, fp16=True):
    """fp32 [rows, d] -> (hi, lo) 16-bit pair [rows, kp] with scale * x = hi + lo (fp16: to 2^-22, bf16: to 2^-17); kp = d padded
    to a multiple of 64 with zero columns."""
    lib = _lib.require_device()
    rows, d = x.shape
    kp = kp or (d + 63) // 64 * 64
    dt = torch.float16 if fp16 else torch.bfloat16
    hi = torch.empty(rows, kp, dtype=dt, device=x.device)
    lo = torch.empty(rows, kp, dtype=dt, device=x.device)
    check(lib.lime_split_bf16_pairs(_ptr(x, torch.float32, "x"), _rowmajor(x, "x"), rows, d, hi.data_ptr(), lo.data_ptr(), kp,
                                    float(scale), 1 if fp16 else 0, _stream()), "lime_split_bf16_pairs")
    return hi, lo


def split_bf16(x, kp=None):
    return split16(x, kp, 1.0, fp16=False)


def cast_bf16(x, kp=None):
    """fp32 [rows, d] (row-major view) -> bf16 [rows, kp], round to nearest, columns d..kp-1 zero (kp = d padded to a multiple
    of 64): the A / W operand of lime_linear_bf16_tma.  lime_split_bf16_pairs with lo = NULL."""
    lib = _lib.require_device()
    rows, d = x.shape
    kp = kp or (d + 63) // 64 * 64
    hi = torch.empty(rows, kp, dtype=torch.bfloat16, device=x.device)
    check(lib.lime_split_bf16_pairs(_ptr(x, torch.float32, "x"), _rowmajor(x, "x"), rows, d, hi.data_ptr(), None, kp,
                                    1.0, 0, _stream()), "lime_split_bf16_pairs")
    return hi


X3_MAX_K = 512
X3_FUSED = True       # linear_x3 as ONE lime_linear_x3_tma launch (False: three accumulating lime_linear_bf16_tma passes)
X3_FUSED_MAX_K = 320  # ... per 320-column slice of the contraction: both W images of a 128-column N tile stay resident (k = 512 in one
                      # launch means 64-column tiles, 5 CTAs pulling every A tile through the L2 path)
X3_ACT_SCALE, X3_W_SCALE = 16.0, 1024.0      # fp16 pairs of the fp32x3 mode: activations * 2^4, weights * 2^10 (hi < 65504, lo out of the subnormals)


def cast_bf16_colsum(x, kp=None):
    """(bf16 image [rows, kp] of x, column sums [d] of x) in one pass over x (lime_cast_bf16_colsum); falls back to cast_bf16 +
    col_sum for shapes the fused kernel does not take."""
    lib = _lib.require_device()
    rows, d = x.shape
    kp = kp or (d + 63) // 64 * 64
    if d % 4 or kp > 1024 or x.stride(0) % 4 or x.data_ptr() % 16 or rows == 0:
        return cast_bf16(x, kp), col_sum(x)
    out16 = torch.empty(rows, kp, dtype=torch.bfloat16, device=x.device)
    cs = torch.zeros(d, dtype=torch.float32, device=x.device)
    check(lib.lime_cast_bf16_colsum(_ptr(x, torch.float32, "x"), _rowmajor(x, "x"), rows, d, out16.data_ptr(), kp,
                                    _ptr(cs, torch.float32, "colsum"), _stream()), "lime_cast_bf16_colsum")
    return out16, cs


def linear_x3(xh, xl, wh, wl, bias=None, residual=None, act=ACT_NONE, out=None, n=None, alpha=1.0):
    """fp32-accurate dense layer on the tensor cores: out = act(alpha x . w^T + bias) + residual with x = xh + xl, w = wh + wl as
    16-bit pairs (fp16: 2^-21 per product; alpha undoes their power-of-two scaling).  X3_FUSED (default): ONE
    lime_linear_x3_tma launch per <= 320-column slice of the contraction (small products and hi.hi in two TMEM accumulators; a
    layer with an activation is one launch up to k = 512); otherwise three accumulating lime_linear_bf16_tma passes (xh.wh
    [+ residual], + xl.wh, + xh.wl + bias then act).  With an activation the residual must be None."""
    assert act == ACT_NONE or residual is None
    n = wh.shape[0] if n is None else n
    kp = xh.shape[1]
    max_k = X3_FUSED_MAX_K if X3_FUSED and act == ACT_NONE else X3_MAX_K      # (a layer with an activation is one launch up to k = 512)
    if kp > max_k:                     # longer contractions accumulate column slices in place (no activation then)
        assert act == ACT_NONE
        for k0 in range(0, kp, max_k):
            k1 = min(kp, k0 + max_k)
            out = linear_x3(xh[:, k0:k1], xl[:, k0:k1], wh[:, k0:k1], wl[:, k0:k1], bias if k0 == 0 else None,
                            residual=residual if k0 == 0 else out, out=out, n=n, alpha=alpha)
        return out
    if X3_FUSED:                       # one launch: the three products accumulate in the same TMEM tile (lime_linear_x3_tma)
        lib = _lib.require_device()
        m = xh.shape[0]
        if out is None:
            out = torch.empty((m, n), dtype=torch.float32, device=xh.device)
        if not (xh.dtype == xl.dtype == wh.dtype == wl.dtype) or xh.dtype not in (torch.bfloat16, torch.float16):
            raise TypeError("operand pairs must all be bfloat16 or all float16")
        lda, ldw = _rowmajor(xh, "xh"), _rowmajor(wh, "wh")
        if _rowmajor(xl, "xl") != lda or _rowmajor(wl, "wl") != ldw or xl.shape != xh.shape or wl.shape != wh.shape:
            raise ValueError("hi / lo images must share shape and row pitch")
        ldr = _rowmajor(residual, "residual") if residual is not None else 0
        check(lib.lime_linear_x3_tma(xh.data_ptr(), xl.data_ptr(), lda, wh.data_ptr(), wl.data_ptr(), ldw,
                                     _ptr(bias, torch.float32, "bias"), _ptr(residual, torch.float32, "residual"), ldr,
                                     _ptr(out, torch.float32, "out"), _rowmajor(out, "out"), m, n, kp, act, float(alpha),
                                     1 if xh.dtype == torch.float16 else 0, _stream()), "lime_linear_x3_tma")
        return out
    out = linear_tma(xh, wh, None, residual=residual, out=out, n=n, out_bf16=False, alpha=alpha)
    linear_tma(xl, wh, None, residual=out, out=out, n=n, out_bf16=False, alpha=alpha)
    linear_tma(xh, wl, bias, residual=out, act=act | ACT_RES_FIRST, out=out, n=n, out_bf16=False, alpha=alpha)
    return out


def linear_x3_pairs(xh, xl, wh, wl, bias=None, act=ACT_NONE, n=None, alpha=1.0, out_scale=1.0):
    """linear_x3 whose result leaves as the next x3 layer's fp16 operand pair: out_scale * act(alpha x . w^T + bias) = hi + lo, each
    [m, kp] (kp = n padded to a multiple of 64, padding columns zero) -- lime_linear_x3_pairs_tma, one launch, k <= 512."""
    lib = _lib.require_device()
    m, kp_in = xh.shape
    n = wh.shape[0] if n is None else n
    kp = (n + 63) // 64 * 64
    hi = torch.empty(m, kp, dtype=torch.float16, device=xh.device)
    lo = torch.empty(m, kp, dtype=torch.float16, device=xh.device)
    if not (xh.dtype == xl.dtype == wh.dtype == wl.dtype == torch.float16):
        raise TypeError("operand pairs must be float16")
    lda, ldw = _rowmajor(xh, "xh"), _rowmajor(wh, "wh")
    if _rowmajor(xl, "xl") != lda or _rowmajor(wl, "wl") != ldw or xl.shape != xh.shape or wl.shape != wh.shape:
        raise ValueError("hi / lo images must share shape and row pitch")
    check(lib.lime_linear_x3_pairs_tma(xh.data_ptr(), xl.data_ptr(), lda, wh.data_ptr(), wl.data_ptr(), ldw,
                                       _ptr(bias, torch.float32, "bias"), hi.data_ptr(), lo.data_ptr(), kp, float(out_scale),
                                       m, n, kp_in, act, float(alpha), 1, _stream()), "lime_linear_x3_pairs_tma")
    return hi, lo


def embed_pe_bf16(E, ids, T, pe, out, out16):
    lib = _lib.require_device()
    check(lib.lime_embed_pe_bf16(_ptr(E, torch.float32, "E"), E.shape[0], _ptr(ids, torch.int32, "ids"), ids.numel(), T,
                                 E.shape[1], _ptr(pe, torch.float32, "pe"), _ptr(out, torch.float32, "out"),
                                 _ptr(out16, torch.bfloat16, "out16"), out16.shape[1], _stream()), "lime_embed_pe_bf16")
    return out, out16


def mha_bf16(qkv16, ctx16, n_news, T, d, nhead):
    lib = _lib.require_device()
    for lo in range(0, n_news, 65535):
        hi = min(n_news, lo + 65535)
        check(lib.lime_mha_bf16(qkv16[lo * T:].data_ptr(), qkv16.stride(0), ctx16[lo * T:].data_ptr(), ctx16.stride(0),
                                hi - lo, T, d, nhead, _stream()), "lime_mha_bf16")
    return ctx16


def layernorm_bf16(x, gamma, beta, out, out16, eps=1e-5):
    lib = _lib.require_device()
    check(lib.lime_layernorm_bf16(_ptr(x, torch.float32, "x"), _rowmajor(x, "x"), _ptr(gamma, torch.float32, "gamma"),
                                  _ptr(beta, torch.float32, "beta"), _ptr(out, torch.float32, "out"), _rowmajor(out, "out"),
                                  _ptr(out16, torch.bfloat16, "out16"), out16.shape[1], x.shape[0], x.shape[1], eps,
                                  _stream()), "lime_layernorm_bf16")
    return out, out16


def _pair_buffers(rows, d, device, kp=None):
    kp = kp or (d + 63) // 64 * 64
    return (torch.empty(rows, kp, dtype=torch.float16, device=device), torch.empty(rows, kp, dtype=torch.float16, device=device))


def embed_pe_pairs(E, ids, T, pe, out, scale):
    """embed_pe + the fp16 operand pair scale * out = hi + lo ([rows, kp], padding columns zero) of the fp32x3 mode."""
    lib = _lib.require_device()
    hi, lo = _pair_buffers(ids.numel(), E.shape[1], out.device)
    check(lib.lime_embed_pe_pairs(_ptr(E, torch.float32, "E"), E.shape[0], _ptr(ids, torch.int32, "ids"), ids.numel(), T,
                                  E.shape[1], _ptr(pe, torch.float32, "pe"), _ptr(out, torch.float32, "out"),
                                  hi.data_ptr(), lo.data_ptr(), hi.shape[1], float(scale), _stream()), "lime_embed_pe_pairs")
    return hi, lo


def layernorm_pairs(x, gamma, beta, out, scale, eps=1e-5):
    """layernorm + the fp16 operand pair scale * out = hi + lo ([rows, kp], padding columns zero) of the fp32x3 mode."""
    lib = _lib.require_device()
    hi, lo = _pair_buffers(x.shape[0], x.shape[1], x.device)
    check(lib.lime_layernorm_pairs(_ptr(x, torch.float32, "x"), _rowmajor(x, "x"), _ptr(gamma, torch.float32, "gamma"),
                                   _ptr(beta, torch.float32, "beta"), _ptr(out, torch.float32, "out"), _rowmajor(out, "out"),
                                   hi.data_ptr(), lo.data_ptr(), hi.shape[1], float(scale), x.shape[0], x.shape[1], eps,
                                   _stream()), "lime_layernorm_pairs")
    return hi, lo


def gemm_strided(a, b, alpha=1.0, out=None):
    """out = alpha * a @ b for arbitrary-stride 2-D views (weight folding only)."""
    lib = _lib.require_device()
    m, k = a.shape
    k2, n = b.shape
    assert k == k2
    if out is None:
        out = torch.empty((m, n), dtype=torch.float32, device=a.device)
    check(lib.lime_gemm_strided(_ptr(a, torch.float32, "a"), a.stride(0), a.stride(1),
                                _ptr(b, torch.float32, "b"), b.stride(0), b.stride(1),
                                _ptr(out, torch.float32, "out"), _rowmajor(out, "out"),
                                m, n, k, float(alpha), _stream()), "lime_gemm_strided")
    return out


def embed_pe(E, ids, T, pe, out):
    lib = _lib.require_device()
    rows = ids.numel()
    check(lib.lime_embed_pe(_ptr(E, torch.float32, "E"), E.shape[0], _ptr(ids, torch.int32, "ids"),
                            rows, T, E.shape[1], _ptr(pe, torch.float32, "pe"),
                            _ptr(out, torch.float32, "out"), _stream()), "lime_embed_pe")
    return out


def mha(qkv, ctx, n_news, T, d, nhead, p_drop=0.0, seed=0, bf16=False, x3=False):
    """attention core; bf16: lime_mha_fwd_bf16 (tensor cores, q k v and P rounded to bf16), the training step's bf16 mode;
    x3: lime_mha_x3 (tensor cores on fp16 hi / lo pairs, fp32-level accuracy), Stage A's fp32x3 mode"""
    lib = _lib.require_device()
    fn = lib.lime_mha_fwd_bf16 if bf16 else lib.lime_mha
    for lo in range(0, n_news, 65535):
        hi = min(n_news, lo + 65535)
        if x3:
            check(lib.lime_mha_x3(qkv[lo * T:].data_ptr(), ctx[lo * T:].data_ptr(), None, None, 0, 1.0, hi - lo, T, d, nhead,
                                  float(p_drop), int(seed) & (2 ** 64 - 1), lo, _stream()), "lime_mha_x3")
        else:
            check(fn(qkv[lo * T:].data_ptr(), ctx[lo * T:].data_ptr(), hi - lo, T, d, nhead, float(p_drop),
                     int(seed) & (2 ** 64 - 1), lo, _stream()), "lime_mha")
    return ctx


def mha_x3_pairs(qkv, n_news, T, d, nhead, scale, kp=None):
    """lime_mha_x3 with the context written as the fp16 operand pair scale * ctx = hi + lo, each [n_news * T, kp] (kp = d padded to
    a multiple of 64, padding columns zero): the A operand of the out_proj linear_x3, no fp32 context and no split pass."""
    lib = _lib.require_device()
    kp = kp or (d + 63) // 64 * 64
    hi16 = torch.empty(n_news * T, kp, dtype=torch.float16, device=qkv.device)
    lo16 = torch.empty(n_news * T, kp, dtype=torch.float16, device=qkv.device)
    for lo in range(0, n_news, 65535):
        hi = min(n_news, lo + 65535)
        check(lib.lime_mha_x3(_ptr(qkv, torch.float32, "qkv") + lo * T * qkv.stride(0) * 4, None, hi16[lo * T:].data_ptr(),
                              lo16[lo * T:].data_ptr(), kp, float(scale), hi - lo, T, d, nhead, 0.0, 0, lo, _stream()), "lime_mha_x3")
    return hi16, lo16


def layernorm(x, gamma, beta, out, eps=1e-5):
    lib = _lib.require_device()
    check(lib.lime_layernorm(_ptr(x, torch.float32, "x"), _rowmajor(x, "x"),
                             _ptr(gamma, torch.float32, "gamma"), _ptr(beta, torch.float32, "beta"),
                             _ptr(out, torch.float32, "out"), _rowmajor(out, "out"), x.shape[0],
                             x.shape[1], eps, _stream()), "lime_layernorm")
    return out


def layernorm_meanpool(x, gamma, beta, out, n_news, T, eps=1e-5):
    """x [n_news*T, d] contiguous -> out[:, :d] (2-D view, any row stride)."""
    lib = _lib.require_device()
    check(lib.lime_layernorm_meanpool(_ptr(x, torch.float32, "x"), _ptr(gamma, torch.float32, "gamma"),
                                      _ptr(beta, torch.float32, "beta"), _ptr(out, torch.float32, "out"),
                                      _rowmajor(out, "out"), n_news, T, x.shape[1], eps, _stream()),
          "lime_layernorm_meanpool")
    return out


def topic_rep(cat_emb, sub_emb, W, b, cat, sub, out, width):
    lib = _lib.require_device()
    check(lib.lime_topic_rep(_ptr(cat_emb, torch.float32, "cat_emb"), _ptr(sub_emb, torch.float32, "sub_emb"),
                             _ptr(W, torch.float32, "W"), _ptr(b, torch.float32, "b"),
                             _ptr(cat, torch.int32, "cat"), _ptr(sub, torch.int32, "sub"), cat.numel(),
                             _ptr(out, torch.float32, "out"), _rowmajor(out, "out"), width, _stream()),
          "lime_topic_rep")
    return out


def intent_pool(pre, e, w2, out, n, k, D):
    lib = _lib.require_device()
    check(lib.lime_intent_pool(_ptr(pre, torch.float32, "pre"), _ptr(e, torch.float32, "e"),
                               _ptr(w2, torch.float32, "w2"), _ptr(out, torch.float32, "out"),
                               _rowmajor(out, "out"), n, k, D, _stream()), "lime_intent_pool")
    return out


def content_fuse(title, body, cat_emb, sub_emb, cat, sub, out):
    lib = _lib.require_device()
    n, D = title.shape
    check(lib.lime_content_fuse(_ptr(title, torch.float32, "title"), _ptr(body, torch.float32, "body"),
                                _ptr(cat_emb, torch.float32, "cat_emb"), _ptr(sub_emb, torch.float32, "sub_emb"),
                                _ptr(cat, torch.int32, "cat"), _ptr(sub, torch.int32, "sub"), n, D,
                                cat_emb.shape[1], sub_emb.shape[1], _ptr(out, torch.float32, "out"),
                                _rowmajor(out, "out"), _stream()), "lime_content_fuse")
    return out


def bucket_pairs(Ef, El, out):
    lib = _lib.require_device()
    check(lib.lime_bucket_pairs(_ptr(Ef, torch.float32, "Ef"), _ptr(El, torch.float32, "El"), Ef.shape[0],
                                Ef.shape[1], _ptr(out, torch.float32, "out"), _stream()), "lime_bucket_pairs")
    return out


def scale_rows(M, row_scale=None, alpha=1.0):
    lib = _lib.require_device()
    check(lib.lime_scale_rows(_ptr(M, torch.float32, "M"), _rowmajor(M, "M"),
                              _ptr(row_scale, torch.float32, "row_scale"), float(alpha), M.shape[0],
                              M.shape[1], _stream()), "lime_scale_rows")
    return M


def prefix_rows(M):
    lib = _lib.require_device()
    check(lib.lime_prefix_rows(_ptr(M, torch.float32, "M"), _rowmajor(M, "M"), M.shape[0], M.shape[1],
                               _stream()), "lime_prefix_rows")
    return M


def rank_metrics(scores, labels, cand_off, want_ranks=True):
    """Per-impression stable ranks (int32 [P]) and [I,4] fp64 (auc, mrr, ndcg5, ndcg10)."""
    lib = _lib.require_device()
    I = cand_off.numel() - 1
    ranks = torch.empty(scores.shape, dtype=torch.int32, device=scores.device) if want_ranks else None
    metrics = torch.empty((I, 4), dtype=torch.float64, device=scores.device)
    check(lib.lime_rank_metrics(_ptr(scores, torch.float32, "scores"), _ptr(labels, torch.uint8, "labels"),
                                _ptr(cand_off, torch.int64, "cand_off"), I,
                                ranks.data_ptr() if want_ranks else None, metrics.data_ptr(), _stream()),
          "lime_rank_metrics")
    return ranks, metrics


TOPK_MAX = 1024      # LIME_TOPK_MAX


def pool_topk(scores, k, pool_index, pool_news=None, exclude=None, hist_news=None, hist_mask=None):
    """lime_pool_topk: scores [U, C] fp32 (row u = user u over the pool positions), pool_index [C] int32 (the id each
    position returns and its tie-break key), optional pool_news [C] int32 + hist_news / hist_mask [U, H] int32 / uint8
    (a position whose news is in the user's masked-in history is never returned), optional exclude [C] uint8.
    -> (index [U, k] int32, -1 padded; score [U, k] fp32, -inf padded; count [U] int32): per user the k largest
    scores, equal scores by ascending pool_index, NaN never returned."""
    lib = _lib.require_device()
    U, C = scores.shape
    if not scores.is_contiguous():
        raise ValueError("scores must be contiguous")
    if pool_index.numel() != C or (pool_news is not None and pool_news.numel() != C) or (exclude is not None and exclude.numel() != C):
        raise ValueError("pool arrays must have one entry per score column")
    H = 0
    if hist_news is not None:
        if hist_mask is None or hist_news.dim() != 2 or hist_news.shape[0] != U or hist_mask.shape != hist_news.shape:
            raise ValueError("hist_news / hist_mask must both be [users, max_history]")
        if not (hist_news.is_contiguous() and hist_mask.is_contiguous()):
            raise ValueError("hist_news / hist_mask must be contiguous")
        H = hist_news.shape[1]
    dev = scores.device
    idx = torch.empty((U, k), dtype=torch.int32, device=dev)
    val = torch.empty((U, k), dtype=torch.float32, device=dev)
    cnt = torch.empty((U,), dtype=torch.int32, device=dev)
    nbytes = int(lib.lime_pool_topk_scratch_bytes(U, C, int(k)))
    scratch = torch.empty((nbytes,), dtype=torch.uint8, device=dev) if nbytes > 0 else None
    check(lib.lime_pool_topk(_ptr(scores, torch.float32, "scores"), U, C, _ptr(pool_index, torch.int32, "pool_index"),
                             _ptr(pool_news, torch.int32, "pool_news"), _ptr(exclude, torch.uint8, "exclude"),
                             _ptr(hist_news, torch.int32, "hist_news"), _ptr(hist_mask, torch.uint8, "hist_mask"), H, int(k),
                             idx.data_ptr(), val.data_ptr(), cnt.data_ptr(),
                             scratch.data_ptr() if scratch is not None else None, _stream()), "lime_pool_topk")
    return idx, val, cnt


POOL_RANK_MAX_TARGETS = 256      # LIME_POOL_RANK_MAX_TARGETS
POOL_RANK_MAX_CUTOFFS = 8        # LIME_POOL_RANK_MAX_CUTOFFS


def pool_rank_metrics(scores, pool_index, target_pos, cutoffs=(), pool_news=None, exclude=None, hist_news=None,
                      hist_mask=None):
    """lime_pool_rank_metrics: scores / pool_index / pool_news / exclude / hist_news / hist_mask as in pool_topk,
    target_pos [U, T] int32 (pool positions of the held-out clicks, -1 = none), cutoffs a host sequence of ints >= 1.
    -> (rank [U, T] int32, 0 = unranked; ranked [U] int32; eligible [U] int64; metrics [U, 4 + 2 len(cutoffs)] fp64 =
    auc, mrr, ndcg5, ndcg10, recall@K, ndcg@K ...): the 1-based position of every target in the order pool_topk
    returns, among every position it could return."""
    lib = _lib.require_device()
    U, C = scores.shape
    if not scores.is_contiguous():
        raise ValueError("scores must be contiguous")
    if pool_index.numel() != C or (pool_news is not None and pool_news.numel() != C) or (exclude is not None and exclude.numel() != C):
        raise ValueError("pool arrays must have one entry per score column")
    if target_pos.dim() != 2 or target_pos.shape[0] != U or not target_pos.is_contiguous():
        raise ValueError("target_pos must be a contiguous [users, targets] tensor")
    H = 0
    if hist_news is not None:
        if hist_mask is None or hist_news.dim() != 2 or hist_news.shape[0] != U or hist_mask.shape != hist_news.shape:
            raise ValueError("hist_news / hist_mask must both be [users, max_history]")
        if not (hist_news.is_contiguous() and hist_mask.is_contiguous()):
            raise ValueError("hist_news / hist_mask must be contiguous")
        H = hist_news.shape[1]
    T = target_pos.shape[1]
    cut = [int(c) for c in cutoffs]
    dev = scores.device
    rank = torch.empty((U, T), dtype=torch.int32, device=dev)
    ranked = torch.empty((U,), dtype=torch.int32, device=dev)
    eligible = torch.empty((U,), dtype=torch.int64, device=dev)
    metrics = torch.empty((U, 4 + 2 * len(cut)), dtype=torch.float64, device=dev)
    scratch = torch.empty((max(1, int(lib.lime_pool_rank_scratch_bytes(U, T))),), dtype=torch.uint8, device=dev)
    h_cut = (ctypes.c_int32 * max(1, len(cut)))(*cut)
    check(lib.lime_pool_rank_metrics(_ptr(scores, torch.float32, "scores"), U, C, _ptr(pool_index, torch.int32, "pool_index"),
                                     _ptr(pool_news, torch.int32, "pool_news"), _ptr(exclude, torch.uint8, "exclude"),
                                     _ptr(hist_news, torch.int32, "hist_news"), _ptr(hist_mask, torch.uint8, "hist_mask"), H,
                                     _ptr(target_pos, torch.int32, "target_pos"), T, h_cut, len(cut), rank.data_ptr(),
                                     ranked.data_ptr(), eligible.data_ptr(), metrics.data_ptr(), scratch.data_ptr(), _stream()),
          "lime_pool_rank_metrics")
    return rank, ranked, eligible, metrics


def metrics_reduce(metrics):
    """[I,4] fp64 -> fp64 [5] = (sum auc, sum mrr, sum ndcg5, sum ndcg10, valid impressions)."""
    lib = _lib.require_device()
    sums = torch.empty(5, dtype=torch.float64, device=metrics.device)
    check(lib.lime_metrics_reduce(_ptr(metrics, torch.float64, "metrics"), metrics.shape[0],
                                  sums.data_ptr(), _stream()), "lime_metrics_reduce")
    return sums


def row_absmax(m, out):
    """out[i] = max_j |m[i, j]| for a 2-D view m; out is a 1-D (possibly strided) view."""
    lib = _lib.require_device()
    check(lib.lime_row_absmax(_ptr(m, torch.float32, "m"), _rowmajor(m, "m"), m.shape[0], m.shape[1],
                              _ptr(out, torch.float32, "out"), out.stride(0), _stream()), "lime_row_absmax")
    return out


CAND16_SCALE = 1024.0      # LIME_CAND16_SCALE


def split_f16_pairs(src, blocks=3, absmax=None, scale=CAND16_SCALE, out=None):
    """lime_split_f16_pairs: fp32 [rows, >= blocks*400] (row-major view) -> fp16 [rows, blocks*800]: the hi halves
    of the ``blocks`` vectors, then their lo halves (operand format of the tensor-core scoring kernel).
    ``absmax``: optional 1-D (strided) fp32 view receiving max |x| per row; ``out``: optional contiguous
    destination (a row range of a larger operand array)."""
    lib = _lib.require_device()
    rows = src.shape[0]
    dst = out if out is not None else torch.empty(rows, blocks * 800, dtype=torch.float16, device=src.device)
    if dst.dtype != torch.float16 or not dst.is_contiguous() or tuple(dst.shape) != (rows, blocks * 800):
        raise _lib.LimeError("split_f16_pairs: out must be a contiguous fp16 [rows, blocks*800] tensor")
    check(lib.lime_split_f16_pairs(_ptr(src, torch.float32, "src"), _rowmajor(src, "src"), rows, blocks, float(scale), dst.data_ptr(),
                                   _ptr(absmax, torch.float32, "absmax") if absmax is not None else None,
                                   absmax.stride(0) if absmax is not None else 0, _stream()), "lime_split_f16_pairs")
    return dst


SCORE_AUTO, SCORE_EXACT, SCORE_FORCE_FALLBACK = 0, 1, 2
_score_mode = SCORE_AUTO


def score_configure(mode=SCORE_AUTO, tolerance=1e-6):
    """lime_score_configure: 0 = tensor-core scoring with exact fallback (default), 1 = exact kernel
    only, 2 = tensor-core path with every unit forced through the fallback (tests)."""
    global _score_mode
    check(_lib.load().lime_score_configure(int(mode), float(tolerance)), "lime_score_configure")
    _score_mode = int(mode)


def score_mode():
    return _score_mode


# ---- training kernels (csrc/train_kernels.cu) -------------------------------------------------------
def gemm(a, a_kmajor, b, b_kmajor, m, n, k, out=None, alpha=1.0, accumulate=False, bf16=False):
    """out[m, n] (+)= alpha * op(a) @ op(b) (lime_gemm / lime_gemm_bf16; see include/lime_b200.h for the layouts)."""
    lib = _lib.require_device()
    if out is None:
        out = torch.empty((m, n), dtype=torch.float32, device=a.device)
    check((lib.lime_gemm_bf16 if bf16 else lib.lime_gemm)(_ptr(a, torch.float32, "a"), _rowmajor(a, "a"), int(bool(a_kmajor)),
                        _ptr(b, torch.float32, "b"), _rowmajor(b, "b"), int(bool(b_kmajor)),
                        _ptr(out, torch.float32, "out"), _rowmajor(out, "out"), m, n, k, float(alpha),
                        int(bool(accumulate)), _stream()), "lime_gemm")
    return out


def gemm_tn_tma(a16, b16, m, n, out=None, alpha=1.0, accumulate=False):
    """out[m, n] (+)= alpha * a16[:, :m].T @ b16[:, :n] over the rows (lime_gemm_bf16_tn_tma): the weight gradient
    dW = dZ^T X on bf16 images [rows, ld] of dZ and X (cast_bf16)."""
    lib = _lib.require_device()
    if a16.dtype != torch.bfloat16 or b16.dtype != torch.bfloat16 or a16.shape[0] != b16.shape[0]:
        raise TypeError("a16 / b16 must be bfloat16 images over the same rows")
    if out is None:
        out = torch.empty((m, n), dtype=torch.float32, device=a16.device)
    check(lib.lime_gemm_bf16_tn_tma(a16.data_ptr(), _rowmajor(a16, "a16"), b16.data_ptr(), _rowmajor(b16, "b16"),
                                    _ptr(out, torch.float32, "out"), _rowmajor(out, "out"), m, n, a16.shape[0], float(alpha),
                                    int(bool(accumulate)), _stream()), "lime_gemm_bf16_tn_tma")
    return out


def act_bwd(dy, y, act, out=None):
    lib = _lib.require_device()
    if out is None:
        out = torch.empty_like(dy)
    check(lib.lime_act_bwd(_ptr(dy, torch.float32, "dy"), _rowmajor(dy, "dy"), _ptr(y, torch.float32, "y"),
                           _rowmajor(y, "y"), _ptr(out, torch.float32, "out"), _rowmajor(out, "out"),
                           dy.shape[0], dy.shape[1], int(act), _stream()), "lime_act_bwd")
    return out


def col_sum(m, out=None):
    lib = _lib.require_device()
    if out is None:
        out = torch.zeros(m.shape[1], dtype=torch.float32, device=m.device)
    check(lib.lime_col_sum(_ptr(m, torch.float32, "m"), _rowmajor(m, "m"), m.shape[0], m.shape[1],
                           _ptr(out, torch.float32, "out"), _stream()), "lime_col_sum")
    return out


def layernorm_bwd(x, gamma, dy, eps=1e-5, bcast_T=0):
    """-> (dx, dgamma, dbeta).  bcast_T > 0: dy has one row per news (mean-pool backward)."""
    lib = _lib.require_device()
    rows, d = x.shape
    dx = torch.empty((rows, d), dtype=torch.float32, device=x.device)
    dg = torch.zeros(d, dtype=torch.float32, device=x.device)
    db = torch.zeros(d, dtype=torch.float32, device=x.device)
    check(lib.lime_layernorm_bwd(_ptr(x, torch.float32, "x"), _rowmajor(x, "x"), _ptr(gamma, torch.float32, "gamma"),
                                 _ptr(dy, torch.float32, "dy"), _rowmajor(dy, "dy"), int(bcast_T), dx.data_ptr(), d,
                                 dg.data_ptr(), db.data_ptr(), rows, d, float(eps), _stream()), "lime_layernorm_bwd")
    return dx, dg, db


def gather_rows(table, ids, out=None):
    lib = _lib.require_device()
    n, d = ids.numel(), table.shape[1]
    if out is None:
        out = torch.empty((n, d), dtype=torch.float32, device=table.device)
    check(lib.lime_gather_rows(_ptr(table, torch.float32, "table"), _rowmajor(table, "table"), table.shape[0],
                               _ptr(ids, torch.int32, "ids"), n, d, _ptr(out, torch.float32, "out"),
                               _rowmajor(out, "out"), _stream()), "lime_gather_rows")
    return out


SCATTER_SORT_MIN = 8192      # id lists at least this long are sorted first (hot rows: pad id, frequent words)


def scatter_add_rows(src, ids, dtable):
    """dtable[ids[r]] += src[r].  Long id lists (the word-embedding gradient) go through lime_scatter_add_rows_sorted:
    torch.sort of the ids (plumbing), then runs of equal ids are summed in registers before one vector reduction."""
    lib = _lib.require_device()
    n, d = ids.numel(), src.shape[1]
    if (n >= SCATTER_SORT_MIN and d % 4 == 0 and d <= 512 and src.stride(0) % 4 == 0 and dtable.stride(0) % 4 == 0
            and src.data_ptr() % 16 == 0 and dtable.data_ptr() % 16 == 0):
        sorted_ids, perm = torch.sort(ids.reshape(-1))
        check(lib.lime_scatter_add_rows_sorted(_ptr(src, torch.float32, "src"), _rowmajor(src, "src"),
                                               _ptr(sorted_ids, torch.int32, "ids"), _ptr(perm, torch.int64, "perm"), n, d,
                                               _ptr(dtable, torch.float32, "dtable"), _rowmajor(dtable, "dtable"),
                                               dtable.shape[0], _stream()), "lime_scatter_add_rows_sorted")
        return dtable
    check(lib.lime_scatter_add_rows(_ptr(src, torch.float32, "src"), _rowmajor(src, "src"),
                                    _ptr(ids, torch.int32, "ids"), ids.numel(), src.shape[1],
                                    _ptr(dtable, torch.float32, "dtable"), _rowmajor(dtable, "dtable"),
                                    dtable.shape[0], _stream()), "lime_scatter_add_rows")
    return dtable


def mha_bwd(qkv, dctx, n_news, T, d, nhead, p_drop=0.0, seed=0, bf16=False):
    """backward of mha; bf16: lime_mha_bwd_bf16 (tensor cores, operands rounded to bf16), the training step's bf16 mode"""
    lib = _lib.require_device()
    dqkv = torch.empty_like(qkv)
    fn = lib.lime_mha_bwd_bf16 if bf16 else lib.lime_mha_bwd
    for lo in range(0, n_news, 65535):
        hi = min(n_news, lo + 65535)
        check(fn(qkv[lo * T:].data_ptr(), dctx[lo * T:].data_ptr(), dqkv[lo * T:].data_ptr(), hi - lo, T, d,
                               nhead, float(p_drop), int(seed) & (2 ** 64 - 1), lo, _stream()), "lime_mha_bwd")
    return dqkv


def intent_pool_bwd(pre, e, w2, dout, n, k, D):
    lib = _lib.require_device()
    dpre, de = torch.empty_like(pre), torch.empty_like(e)
    dw2 = torch.zeros(D, dtype=torch.float32, device=pre.device)
    check(lib.lime_intent_pool_bwd(_ptr(pre, torch.float32, "pre"), _ptr(e, torch.float32, "e"), _ptr(w2, torch.float32, "w2"),
                                   _ptr(dout, torch.float32, "dout"), _rowmajor(dout, "dout"), dpre.data_ptr(), de.data_ptr(),
                                   dw2.data_ptr(), n, k, D, _stream()), "lime_intent_pool_bwd")
    return dpre, de, dw2


def content_fuse_bwd(title, body, dcontent):
    lib = _lib.require_device()
    n, D = title.shape
    dt, db = torch.empty_like(title), torch.empty_like(body)
    check(lib.lime_content_fuse_bwd(_ptr(title, torch.float32, "title"), _ptr(body, torch.float32, "body"),
                                    _ptr(dcontent, torch.float32, "dcontent"), _rowmajor(dcontent, "dcontent"), n, D,
                                    dt.data_ptr(), db.data_ptr(), _stream()), "lime_content_fuse_bwd")
    return dt, db


def dropout(x, p, seed, out=None):
    """y = x * keep / (1 - p) with a stateless mask (same call on the gradient = backward)."""
    lib = _lib.require_device()
    if out is None:
        out = torch.empty_like(x)
    check(lib.lime_dropout(_ptr(x, torch.float32, "x"), _rowmajor(x, "x"), _ptr(out, torch.float32, "out"),
                           _rowmajor(out, "out"), x.shape[0], x.shape[1], float(p), int(seed) & (2 ** 64 - 1), _stream()),
          "lime_dropout")
    return out


_M64 = 2 ** 64 - 1


def dropout_fused(x, p, seed, res=None, seed2=None):
    """x * m(seed) [* m(seed2)] [+ res] in one pass (lime_dropout_fused), the masks of ``dropout``."""
    lib = _lib.require_device()
    out = torch.empty_like(x)
    check(lib.lime_dropout_fused(_ptr(x, torch.float32, "x"), _rowmajor(x, "x"), _ptr(res, torch.float32, "res"),
                                 _rowmajor(res, "res") if res is not None else 0, _ptr(out, torch.float32, "out"),
                                 _rowmajor(out, "out"), x.shape[0], x.shape[1], float(p), int(seed) & _M64,
                                 int(seed2 or 0) & _M64, 0 if seed2 is None else 1, _stream()), "lime_dropout_fused")
    return out


def embed_pe_dropout(E, ids, T, pe, p, seed_w, seed_x):
    """m_x * (m_w * E[ids] + pe) -> [ids.numel(), d] (lime_embed_pe_dropout)."""
    lib = _lib.require_device()
    out = torch.empty((ids.numel(), E.shape[1]), dtype=torch.float32, device=E.device)
    check(lib.lime_embed_pe_dropout(_ptr(E, torch.float32, "E"), E.shape[0], _ptr(ids, torch.int32, "ids"), ids.numel(), int(T),
                                    E.shape[1], _ptr(pe, torch.float32, "pe"), float(p), int(seed_w) & _M64, int(seed_x) & _M64,
                                    _ptr(out, torch.float32, "out"), _stream()), "lime_embed_pe_dropout")
    return out


# ---- training kernels of the user encoder (csrc/train_user.cu) -------------------------------------
def _f32(t, name):
    return _ptr(t, torch.float32, name)


def ca_attention_fwd(Qp, Kp, mask, B, N, H, p_drop=0.0, seed=0):
    lib = _lib.require_device()
    a = torch.empty((B * H,), dtype=torch.float32, device=Qp.device)
    check(lib.lime_ca_attention_fwd(_f32(Qp, "Qp"), _f32(Kp, "Kp"), _ptr(mask, torch.uint8, "mask"), B, N, H,
                                    float(p_drop), int(seed) & (2 ** 64 - 1), a.data_ptr(), _stream()), "lime_ca_attention_fwd")
    return a


def ca_attention_bwd(Qp, Kp, mask, B, N, H, da, p_drop=0.0, seed=0):
    lib = _lib.require_device()
    dQ, dK = torch.empty_like(Qp), torch.empty_like(Kp)
    check(lib.lime_ca_attention_bwd(_f32(Qp, "Qp"), _f32(Kp, "Kp"), _ptr(mask, torch.uint8, "mask"), B, N, H,
                                    float(p_drop), int(seed) & (2 ** 64 - 1), _f32(da, "da"),
                                    dQ.data_ptr(), dK.data_ptr(), _stream()), "lime_ca_attention_bwd")
    return dQ, dK


def row_scale_fwd(v, a):
    lib = _lib.require_device()
    out = torch.empty_like(v)
    check(lib.lime_row_scale_fwd(_f32(v, "v"), _f32(a, "a"), v.shape[0], v.shape[1], out.data_ptr(), _stream()), "lime_row_scale_fwd")
    return out


def row_scale_bwd(v, a, dwc):
    lib = _lib.require_device()
    dv, da = torch.empty_like(v), torch.empty_like(a)
    check(lib.lime_row_scale_bwd(_f32(v, "v"), _f32(a, "a"), _f32(dwc, "dwc"), v.shape[0], v.shape[1], dv.data_ptr(),
                                 da.data_ptr(), _stream()), "lime_row_scale_bwd")
    return dv, da


def gate_mix_fwd(z, wc, v):
    lib = _lib.require_device()
    o = torch.empty_like(v)
    check(lib.lime_gate_mix_fwd(_f32(z, "z"), _f32(wc, "wc"), _f32(v, "v"), v.numel(), o.data_ptr(), _stream()), "lime_gate_mix_fwd")
    return o


def gate_mix_bwd(z, wc, v, dout):
    lib = _lib.require_device()
    dz, dwc, dv = torch.empty_like(v), torch.empty_like(v), torch.empty_like(v)
    check(lib.lime_gate_mix_bwd(_f32(z, "z"), _f32(wc, "wc"), _f32(v, "v"), _f32(dout, "dout"), v.numel(), dz.data_ptr(),
                                dwc.data_ptr(), dv.data_ptr(), _stream()), "lime_gate_mix_bwd")
    return dz, dwc, dv


def sage_mean_fwd(x, un, B, H, P):
    lib = _lib.require_device()
    m = torch.empty((B, x.shape[1]), dtype=torch.float32, device=x.device)
    check(lib.lime_sage_mean_fwd(_f32(x, "x"), _f32(un, "un"), B, H, P, un.shape[0], m.data_ptr(), _stream()), "lime_sage_mean_fwd")
    return m


def sage_mean_bwd(dm, B, H, P, un_rows):
    lib = _lib.require_device()
    d = dm.shape[1]
    dx = torch.empty((B * H, d), dtype=torch.float32, device=dm.device)
    dun = torch.empty((un_rows, d), dtype=torch.float32, device=dm.device)
    check(lib.lime_sage_mean_bwd(_f32(dm, "dm"), B, H, P, un_rows, dx.data_ptr(), dun.data_ptr(), _stream()), "lime_sage_mean_bwd")
    return dx, dun


def add_row_bcast(r, l, H):
    lib = _lib.require_device()
    g = torch.empty_like(r)
    check(lib.lime_add_row_bcast(_f32(r, "r"), _f32(l, "l"), r.shape[0], H, r.shape[1], g.data_ptr(), _stream()), "lime_add_row_bcast")
    return g


def sum_over_h(dg, B, H):
    lib = _lib.require_device()
    dl = torch.empty((B, dg.shape[1]), dtype=torch.float32, device=dg.device)
    check(lib.lime_sum_over_h(_f32(dg, "dg"), B, H, dg.shape[1], dl.data_ptr(), _stream()), "lime_sum_over_h")
    return dl


def pool_fwd(Kg, q, g, B, N, H):
    lib = _lib.require_device()
    u = torch.empty((B * N, Kg.shape[1]), dtype=torch.float32, device=Kg.device)
    alpha = torch.empty((B * N, H), dtype=torch.float32, device=Kg.device)
    check(lib.lime_pool_fwd(_f32(Kg, "Kg"), _f32(q, "q"), _f32(g, "g"), B, N, H, u.data_ptr(), alpha.data_ptr(), _stream()),
          "lime_pool_fwd")
    return u, alpha


def pool_bwd(Kg, q, g, alpha, du, B, N, H):
    lib = _lib.require_device()
    dKg, dq, dg = torch.empty_like(Kg), torch.empty_like(q), torch.empty_like(g)
    check(lib.lime_pool_bwd(_f32(Kg, "Kg"), _f32(q, "q"), _f32(g, "g"), _f32(alpha, "alpha"), _f32(du, "du"), B, N, H,
                            dKg.data_ptr(), dq.data_ptr(), dg.data_ptr(), _stream()), "lime_pool_bwd")
    return dKg, dq, dg


def click_score_fwd(u, c, remaining, alpha, beta, use_weighting, use_penalty):
    lib = _lib.require_device()
    rows = u.shape[0]
    s = torch.empty((rows,), dtype=torch.float32, device=u.device)
    w = torch.empty((rows,), dtype=torch.float32, device=u.device)
    check(lib.lime_click_score_fwd(_f32(u, "u"), _f32(c, "c"), _f32(remaining, "remaining"), rows, float(alpha), float(beta),
                                   int(bool(use_weighting)), int(bool(use_penalty)), s.data_ptr(), w.data_ptr(), _stream()),
          "lime_click_score_fwd")
    return s, w


def click_score_bwd(u, c, w, ds):
    lib = _lib.require_device()
    du, dc = torch.empty_like(u), torch.empty_like(c)
    check(lib.lime_click_score_bwd(_f32(u, "u"), _f32(c, "c"), _f32(w, "w"), _f32(ds, "ds"), u.shape[0], du.data_ptr(),
                                   dc.data_ptr(), _stream()), "lime_click_score_bwd")
    return du, dc
