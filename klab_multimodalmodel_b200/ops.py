"""Thin torch-tensor wrappers over the C ABI (include/klab_b200.h).

PyTorch is used here only for device memory and streams: every arithmetic step is a kernel of
libklab_b200.so launched on torch's current CUDA stream.  Nothing in this module falls back to torch ops.
"""
from __future__ import annotations

import ctypes as C
import math

import torch

from . import _lib as L

_DT = {torch.float32: L.F32, torch.bfloat16: L.BF16}


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


def _bytes(n: int, device) -> torch.Tensor:
    return torch.empty(max(int(n), 16), dtype=torch.uint8, device=device)


def launch_count() -> int:
    return int(L.lib().klab_launch_count())


def sm_reserve_info() -> dict:
    return {"sm_budget": int(L.lib().klab_sm_budget())}


# ------------------------------------------------------------------------------------------------
# GEMM
# ------------------------------------------------------------------------------------------------
def gemm(a: torch.Tensor, b: torch.Tensor, M: int, N: int, K: int, *, a_mn: bool = False, b_mn: bool = False,
         out: torch.Tensor | None = None, out_dtype: torch.dtype | None = None, bias: torch.Tensor | None = None,
         act: int = L.ACT_NONE, residual: torch.Tensor | None = None, aux_in: torch.Tensor | None = None,
         aux_out: torch.Tensor | None = None, alpha: float = 1.0, accumulate: bool = False,
         dropout_p: float = 0.0, seed: int = 0, seed_ptr: torch.Tensor | None = None, ldd_pad: int | None = None) -> torch.Tensor:
    """D[M,N] = epilogue(alpha * A(m,k) B(n,k)); see klab_gemm in include/klab_b200.h.

    `a` / `b` are 2-D tensors whose row stride is taken from .stride(0) (column slices of a wider buffer are fine).
    """
    assert a.dtype == b.dtype and a.dtype in _DT, (a.dtype, b.dtype)
    assert a.stride(1) == 1 and b.stride(1) == 1
    if out is None:
        od = out_dtype or a.dtype
        if ldd_pad is not None:
            out = torch.empty(M, ldd_pad, dtype=od, device=a.device)[:, :N]
        else:
            out = torch.empty(M, N, dtype=od, device=a.device)
    assert out.stride(1) == 1
    e = L.GemmEpilogue()
    e.bias = _p(bias)
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.numel() == N
    e.residual = _p(residual)
    e.aux_in = _p(aux_in)
    e.aux_out = _p(aux_out)
    e.ldr = residual.stride(0) if residual is not None else 0
    e.ld_aux_in = aux_in.stride(0) if aux_in is not None else 0
    e.ld_aux_out = aux_out.stride(0) if aux_out is not None else 0
    e.alpha = alpha
    e.act = act
    e.accumulate = int(accumulate)
    e.out_dtype = _DT[out.dtype]
    e.res_dtype = _DT[residual.dtype] if residual is not None else 0
    e.aux_in_dtype = _DT[aux_in.dtype] if aux_in is not None else 0
    if aux_out is not None:
        assert aux_out.dtype == out.dtype
    e.dropout_p = dropout_p
    e.dropout_seed = seed
    e.dropout_seed_ptr = _p(seed_ptr)
    if _GEMM_CHECK and a.dtype == torch.bfloat16:
        _gemm_cross_check(a, b, M, N, K, a_mn, b_mn, out, e, aux_out)
    L.check(L.lib().klab_gemm(_stream(), _DT[a.dtype], M, N, K, a.data_ptr(), a.stride(0), int(a_mn),
                              b.data_ptr(), b.stride(0), int(b_mn), out.data_ptr(), out.stride(0), C.byref(e)))
    if _GEMM_CHECK and a.dtype == torch.bfloat16:
        _gemm_cross_check_finish(out, M, N, K, a_mn, b_mn, e)
    return out


# KLAB_GEMM_CHECK=1: run every bf16 tcgen05 GEMM a second time on the fp32-accumulating SIMT kernel (same operands, same
# epilogue) and report the calls whose results differ -- an on-device self check, not a fallback.
import os as _os
_GEMM_CHECK = bool(int(_os.environ.get("KLAB_GEMM_CHECK", "0")))
_check_state: dict = {}


def _gemm_cross_check(a, b, M, N, K, a_mn, b_mn, out, e, aux_out):
    import copy
    ref = out.clone() if e.accumulate else torch.empty_like(out)
    e2 = L.GemmEpilogue()
    C.memmove(C.byref(e2), C.byref(e), C.sizeof(e))
    if aux_out is not None:
        e2.aux_out = None
    L.check(L.lib().klab_gemm_simt(_stream(), _DT[a.dtype], M, N, K, a.data_ptr(), a.stride(0), int(a_mn), b.data_ptr(),
                                   b.stride(0), int(b_mn), ref.data_ptr(), ref.stride(0), C.byref(e2)))
    _check_state["ref"] = ref


def _gemm_cross_check_finish(out, M, N, K, a_mn, b_mn, e):
    ref = _check_state.pop("ref")
    o, r = out.float(), ref.float()
    err = (o - r).abs().max().item()
    scale = r.abs().max().item()
    bad = not (err <= 2e-2 * scale + 1e-6)
    _check_state["n"] = _check_state.get("n", 0) + 1
    if bad:
        print(f"[KLAB_GEMM_CHECK] call #{_check_state['n']} MISMATCH M={M} N={N} K={K} a_mn={int(a_mn)} b_mn={int(b_mn)} act={e.act} "
              f"alpha={e.alpha:.4f} acc={e.accumulate} out_dtype={e.out_dtype} bias={bool(e.bias)} res={bool(e.residual)} "
              f"ldd={out.stride(0)}: max err {err:.3e} vs scale {scale:.3e}", flush=True)


def linear_fwd(x, w, **kw):
    """y[M,N] = x[M,K] w[N,K]^T"""
    return gemm(x, w, x.shape[0], w.shape[0], x.shape[1], **kw)


def linear_dgrad(dy, w, **kw):
    """dx[M,K] = dy[M,N] w[N,K]"""
    return gemm(dy, w, dy.shape[0], w.shape[1], dy.shape[1], b_mn=True, **kw)


def linear_wgrad(dy, x, **kw):
    """dw[N,K] = dy[M,N]^T x[M,K]  (fp32 output: master-weight gradient)"""
    kw.setdefault("out_dtype", torch.float32)
    return gemm(dy, x, dy.shape[1], x.shape[1], dy.shape[0], a_mn=True, b_mn=True, **kw)


# ------------------------------------------------------------------------------------------------
# norms / reductions
# ------------------------------------------------------------------------------------------------
def rmsnorm_fwd(x, gamma, eps, *, out=None, out_rows_per_group=0, out_group_stride=0, save_stats=True):
    rows, d = x.shape
    y = torch.empty(rows, d, dtype=x.dtype, device=x.device) if out is None else out
    rstd = torch.empty(rows, dtype=torch.float32, device=x.device) if save_stats else None
    ldy = y.stride(0) if out is None else out.stride(-2)
    L.check(L.lib().klab_rmsnorm_fwd(_stream(), _DT[x.dtype], rows, d, x.data_ptr(), x.stride(0), gamma.data_ptr(), eps,
                                     y.data_ptr(), ldy, out_rows_per_group, out_group_stride, _p(rstd)))
    return y, rstd


def rmsnorm_bwd(dy, x, gamma, rstd, dres=None, dgamma=None, drop=None, dgamma_out=None):
    """-> (dx, dgamma), or (dx, dgamma, dropout(dx)) with drop = (p, seed, seed_ptr): the mask `dropout_apply` would draw.
    dgamma given: the gain gradient is ACCUMULATED into it; dgamma_out given: it is WRITTEN there (a slice of a flat gradient buffer)."""
    rows, d = x.shape
    dx = torch.empty(rows, d, dtype=x.dtype, device=x.device)
    acc = dgamma is not None
    if dgamma is None:
        dgamma = dgamma_out if dgamma_out is not None else torch.empty(d, dtype=torch.float32, device=x.device)
    ws = _bytes(L.lib().klab_norm_bwd_workspace_bytes(rows, d), x.device)
    if drop is not None and drop[0] > 0.0:
        p, seed, seed_ptr = drop
        dxd = torch.empty(rows, d, dtype=x.dtype, device=x.device)
        L.check(L.lib().klab_rmsnorm_bwd_dropout(_stream(), _DT[x.dtype], rows, d, dy.data_ptr(), dy.stride(0), x.data_ptr(), x.stride(0),
                                                 gamma.data_ptr(), rstd.data_ptr(), _p(dres), dres.stride(0) if dres is not None else 0,
                                                 dx.data_ptr(), dx.stride(0), dgamma.data_ptr(), int(acc), ws.data_ptr(), dxd.data_ptr(),
                                                 float(p), int(seed), _p(seed_ptr)))
        return dx, dgamma, dxd
    L.check(L.lib().klab_rmsnorm_bwd(_stream(), _DT[x.dtype], rows, d, dy.data_ptr(), dy.stride(0), x.data_ptr(), x.stride(0),
                                     gamma.data_ptr(), rstd.data_ptr(), _p(dres), dres.stride(0) if dres is not None else 0,
                                     dx.data_ptr(), dx.stride(0), dgamma.data_ptr(), int(acc), ws.data_ptr()))
    if drop is not None:
        return dx, dgamma, dx
    return dx, dgamma


def layernorm_fwd(x, gamma, beta, eps, residual=None, *, out=None, out_rows_per_group=0, out_group_stride=0, save_stats=True):
    rows, d = x.shape
    y = torch.empty(rows, d, dtype=x.dtype, device=x.device) if out is None else out
    mean = torch.empty(rows, dtype=torch.float32, device=x.device) if save_stats else None
    rstd = torch.empty(rows, dtype=torch.float32, device=x.device) if save_stats else None
    ldy = y.stride(0) if out is None else out.stride(-2)
    L.check(L.lib().klab_layernorm_fwd(_stream(), _DT[x.dtype], rows, d, x.data_ptr(), x.stride(0), gamma.data_ptr(), beta.data_ptr(),
                                       eps, _p(residual), residual.stride(0) if residual is not None else 0, y.data_ptr(), ldy,
                                       out_rows_per_group, out_group_stride, _p(mean), _p(rstd)))
    return y, mean, rstd


def layernorm_bwd(dy, x, gamma, mean, rstd, dres=None, *, dy_ld=None, dy_rows_per_group=0, dy_group_stride=0, dgamma=None, dbeta=None,
                  accumulate=True):
    """dgamma / dbeta given (both or neither): the parameter gradients are accumulated into them (`accumulate`) or written there."""
    rows, d = x.shape
    dx = torch.empty(rows, d, dtype=x.dtype, device=x.device)
    given = dgamma is not None
    assert given == (dbeta is not None)
    acc = given and accumulate
    if not given:
        dgamma = torch.empty(d, dtype=torch.float32, device=x.device)
        dbeta = torch.empty(d, dtype=torch.float32, device=x.device)
    ws = _bytes(L.lib().klab_norm_bwd_workspace_bytes(rows, d), x.device)
    L.check(L.lib().klab_layernorm_bwd(_stream(), _DT[x.dtype], rows, d, dy.data_ptr(), dy.stride(0) if dy_ld is None else dy_ld,
                                       dy_rows_per_group, dy_group_stride, x.data_ptr(), x.stride(0), gamma.data_ptr(),
                                       mean.data_ptr(), rstd.data_ptr(), _p(dres), dres.stride(0) if dres is not None else 0,
                                       dx.data_ptr(), dx.stride(0), dgamma.data_ptr(), dbeta.data_ptr(), int(acc), ws.data_ptr()))
    return dx, dgamma, dbeta


def colsum(x, out=None, accumulate=True):
    """out given: the column sums are accumulated into it (`accumulate`) or written there."""
    rows, d = x.shape
    acc = out is not None and accumulate
    if out is None:
        out = torch.empty(d, dtype=torch.float32, device=x.device)
    ws = _bytes(L.lib().klab_colsum_workspace_bytes(rows, d), x.device)
    L.check(L.lib().klab_colsum(_stream(), _DT[x.dtype], rows, d, x.data_ptr(), x.stride(0), out.data_ptr(), int(acc), ws.data_ptr()))
    return out


# ------------------------------------------------------------------------------------------------
# T5 attention
# ------------------------------------------------------------------------------------------------
def t5_rel_bucket_lut(lq: int, lk: int, bidirectional: bool, num_buckets: int, max_distance: int, q_offset: int = 0):
    """int32 LUT of T5Attention._relative_position_bucket (HF/models/t5/modeling_t5.py:189-234) for every relative
    position r = j - (i + q_offset) that can occur, index r + rel_zero.  Computed on the host with the same torch
    ops (fp32 log, truncation) as the reference so the bucket edges are bit-identical."""
    lo = -(lq - 1 + q_offset)
    rel = torch.arange(lo, lk, dtype=torch.long)
    nb = num_buckets
    buckets = torch.zeros_like(rel)
    if bidirectional:
        nb //= 2
        buckets = buckets + (rel > 0).to(torch.long) * nb
        rel = torch.abs(rel)
    else:
        rel = -torch.min(rel, torch.zeros_like(rel))
    max_exact = nb // 2
    is_small = rel < max_exact
    large = max_exact + (torch.log(rel.float() / max_exact) / math.log(max_distance / max_exact) * (nb - max_exact)).to(torch.long)
    large = torch.min(large, torch.full_like(large, nb - 1))
    buckets = buckets + torch.where(is_small, rel, large)
    return buckets.to(torch.int32), -lo


def t5_attention_fwd(q, k, v, B, H, Lq, Lk, dk, *, bias_table=None, lut=None, rel_zero=0, num_buckets=32, causal=False,
                     q_offset=0, dropout_p=0.0, seed=0, seed_ptr=None, out=None):
    ctx = torch.empty(B * Lq, H * dk, dtype=q.dtype, device=q.device) if out is None else out
    lse = torch.empty(B, H, Lq, dtype=torch.float32, device=q.device)
    L.check(L.lib().klab_t5_attention_fwd(_stream(), _DT[q.dtype], B, H, Lq, Lk, dk, q.data_ptr(), q.stride(0), k.data_ptr(),
                                          k.stride(0), v.data_ptr(), v.stride(0), ctx.data_ptr(), ctx.stride(0), _p(bias_table),
                                          _p(lut), rel_zero, num_buckets, int(causal), q_offset, lse.data_ptr(), dropout_p, seed,
                                          _p(seed_ptr)))
    return ctx, lse


def t5_attention_decode_beam(q, k, v, rows, H, Lk, dk, *, kv_group, src=None, bias_table=None, lut=None, rel_zero=0, q_offset=0,
                             out=None):
    """One query row per hypothesis: self-attention through the ancestry table `src` [rows, ld] int32, or (src None)
    cross-attention where `kv_group` consecutive rows share one sample's Lk K/V rows."""
    ctx = torch.empty(rows, H * dk, dtype=q.dtype, device=q.device) if out is None else out
    L.check(L.lib().klab_t5_attention_decode_beam(_stream(), _DT[q.dtype], rows, H, Lk, dk, q.data_ptr(), q.stride(0), k.data_ptr(),
                                                  k.stride(0), v.data_ptr(), v.stride(0), ctx.data_ptr(), ctx.stride(0), kv_group,
                                                  _p(src), 0 if src is None else src.stride(0), _p(bias_table), _p(lut), rel_zero,
                                                  q_offset))
    return ctx


def t5_attention_bwd(q, k, v, ctx, dctx, lse, dq, dk_, dv, B, H, Lq, Lk, dk, *, bias_table=None, lut=None, rel_zero=0,
                     num_buckets=32, causal=False, q_offset=0, dbias_table=None, dropout_p=0.0, seed=0, seed_ptr=None):
    """dq / dk_ / dv are preallocated outputs with the same row strides as q / k / v."""
    assert dq.stride(0) == q.stride(0) and dk_.stride(0) == k.stride(0) and dv.stride(0) == v.stride(0)
    assert dctx.stride(0) == ctx.stride(0)
    ws = _bytes(L.lib().klab_t5_attention_bwd_workspace_bytes(B, H, Lq, num_buckets), q.device)
    L.check(L.lib().klab_t5_attention_bwd(_stream(), _DT[q.dtype], B, H, Lq, Lk, dk, q.data_ptr(), q.stride(0), k.data_ptr(),
                                          k.stride(0), v.data_ptr(), v.stride(0), ctx.data_ptr(), dctx.data_ptr(), ctx.stride(0),
                                          dq.data_ptr(), dk_.data_ptr(), dv.data_ptr(), _p(bias_table), _p(lut), rel_zero,
                                          num_buckets, int(causal), q_offset, lse.data_ptr(), _p(dbias_table), dropout_p, seed,
                                          _p(seed_ptr), ws.data_ptr()))


# ------------------------------------------------------------------------------------------------
# Swin-V2 window attention
# ------------------------------------------------------------------------------------------------
def swin_tables(window: int, pretrained_window: int):
    """relative_coords_table ((2w-1)^2, 2) fp32 and relative_position_index (N, N) int32, built with the reference's own
    torch ops (HF/models/swinv2/modeling_swinv2.py:489-524)."""
    w = window
    r = torch.arange(-(w - 1), w, dtype=torch.int64).float()
    t = torch.stack(torch.meshgrid([r, r], indexing="ij")).permute(1, 2, 0).contiguous().unsqueeze(0)
    if pretrained_window > 0:
        t[:, :, :, 0] /= pretrained_window - 1
        t[:, :, :, 1] /= pretrained_window - 1
    elif w > 1:
        t[:, :, :, 0] /= w - 1
        t[:, :, :, 1] /= w - 1
    t *= 8
    t = torch.sign(t) * torch.log2(torch.abs(t) + 1.0) / math.log2(8)
    c = torch.stack(torch.meshgrid([torch.arange(w), torch.arange(w)], indexing="ij")).flatten(1)
    rel = (c[:, :, None] - c[:, None, :]).permute(1, 2, 0).contiguous()
    rel[:, :, 0] += w - 1
    rel[:, :, 1] += w - 1
    rel[:, :, 0] *= 2 * w - 1
    return t.view(-1, 2).contiguous().float(), rel.sum(-1).to(torch.int32).contiguous()


def swin_cpb_fwd(coords, index, w1, b1, w2, heads, n_tokens):
    T, U = coords.shape[0], w1.shape[0]
    dev = coords.device
    hidden = torch.empty(T, U, dtype=torch.float32, device=dev)
    tab = torch.empty(T, heads, dtype=torch.float32, device=dev)
    bias = torch.empty(heads, n_tokens, n_tokens, dtype=torch.float32, device=dev)
    L.check(L.lib().klab_swin_cpb_fwd(_stream(), T, U, heads, n_tokens, coords.data_ptr(), index.data_ptr(), w1.data_ptr(),
                                      b1.data_ptr(), w2.data_ptr(), hidden.data_ptr(), tab.data_ptr(), bias.data_ptr()))
    return bias, hidden, tab


def swin_cpb_bwd(coords, index, w2, hidden, tab, dbias, heads, n_tokens, acc_into=None, out=None):
    """acc_into = (dw1, db1, dw2): the gradients are ACCUMULATED into these tensors; out = (dw1, db1, dw2): they are WRITTEN there;
    neither: freshly allocated."""
    T, U = coords.shape[0], hidden.shape[1]
    dev = coords.device
    dtab = torch.empty(T, heads, dtype=torch.float32, device=dev)
    if acc_into is not None:
        dw1, db1, dw2 = acc_into
    elif out is not None:
        dw1, db1, dw2 = out
    else:
        dw1 = torch.empty(U, 2, dtype=torch.float32, device=dev)
        db1 = torch.empty(U, dtype=torch.float32, device=dev)
        dw2 = torch.empty(heads, U, dtype=torch.float32, device=dev)
    L.check(L.lib().klab_swin_cpb_bwd(_stream(), T, U, heads, n_tokens, coords.data_ptr(), index.data_ptr(), w2.data_ptr(),
                                      hidden.data_ptr(), tab.data_ptr(), dbias.data_ptr(), dtab.data_ptr(), dw1.data_ptr(),
                                      db1.data_ptr(), dw2.data_ptr(), int(acc_into is not None)))
    return dw1, db1, dw2


def swin_attention_fwd(q, k, v, B, res, heads, hd, window, shift, logit_scale, bias):
    n = window * window
    nw = (res // window) ** 2
    ctx = torch.empty(B * res * res, heads * hd, dtype=q.dtype, device=q.device)
    lse = torch.empty(B * nw, heads, n, dtype=torch.float32, device=q.device)
    assert q.stride(0) == k.stride(0) == v.stride(0)
    L.check(L.lib().klab_swin_attention_fwd(_stream(), _DT[q.dtype], B, res, heads, hd, window, shift, q.data_ptr(), k.data_ptr(),
                                            v.data_ptr(), q.stride(0), ctx.data_ptr(), ctx.stride(0), logit_scale.data_ptr(),
                                            bias.data_ptr(), lse.data_ptr()))
    return ctx, lse


def swin_attention_bwd(q, k, v, ctx, dctx, dq, dk, dv, B, res, heads, hd, window, shift, logit_scale, bias, lse, dls_out=None):
    n = window * window
    assert dq.stride(0) == q.stride(0) == dk.stride(0) == dv.stride(0) and dctx.stride(0) == ctx.stride(0)
    dbias = torch.empty(heads, n, n, dtype=torch.float32, device=q.device)
    dls = torch.empty(heads, dtype=torch.float32, device=q.device) if dls_out is None else dls_out
    L.check(L.lib().klab_swin_attention_bwd(_stream(), _DT[q.dtype], B, res, heads, hd, window, shift, q.data_ptr(), k.data_ptr(),
                                            v.data_ptr(), q.stride(0), ctx.data_ptr(), dctx.data_ptr(), ctx.stride(0), dq.data_ptr(),
                                            dk.data_ptr(), dv.data_ptr(), logit_scale.data_ptr(), bias.data_ptr(), lse.data_ptr(),
                                            dbias.data_ptr(), dls.data_ptr()))
    return dbias, dls


# ------------------------------------------------------------------------------------------------
# embeddings, patch ops, cross entropy, casts
# ------------------------------------------------------------------------------------------------
_err_flags: dict = {}


def err_flag(device) -> torch.Tensor:
    """Per-device int32 flag the kernels raise on out-of-range token ids / labels (checked by `check_err_flag`)."""
    key = (device.type, device.index)
    if key not in _err_flags:
        _err_flags[key] = torch.zeros(1, dtype=torch.int32, device=device)
    return _err_flags[key]


def check_err_flag(device) -> None:
    f = err_flag(device)
    v = int(f.item())
    if v:
        f.zero_()
        raise IndexError("token id out of range of the embedding table" if v == 1 else "label out of range of the vocabulary")


def embedding_fwd(ids, table, *, shift_right=False, start_id=0, pad_id=0, out=None):
    B, Lx = ids.shape
    vocab, d = table.shape
    y = torch.empty(B * Lx, d, dtype=table.dtype, device=table.device) if out is None else out
    assert ids.dtype == torch.int64 and ids.is_contiguous()
    L.check(L.lib().klab_embedding_fwd(_stream(), _DT[table.dtype], B, Lx, ids.data_ptr(), int(shift_right), start_id, pad_id,
                                       table.data_ptr(), vocab, d, y.data_ptr(), y.stride(0), err_flag(table.device).data_ptr()))
    return y


def embedding_bwd(ids, dout, dtable, *, shift_right=False, start_id=0, pad_id=0):
    B, Lx = ids.shape
    vocab, d = dtable.shape
    assert dtable.dtype == torch.float32 and dtable.is_contiguous()
    L.check(L.lib().klab_embedding_bwd(_stream(), _DT[dout.dtype], B, Lx, ids.data_ptr(), int(shift_right), start_id, pad_id,
                                       dout.data_ptr(), dout.stride(0), d, dtable.data_ptr(), vocab))


def patchify(pixels, patch, dtype):
    B, Cc, H, W = pixels.shape
    assert pixels.dtype == torch.float32 and pixels.is_contiguous()
    out = torch.empty(B * (H // patch) * (W // patch), Cc * patch * patch, dtype=dtype, device=pixels.device)
    L.check(L.lib().klab_patchify(_stream(), _DT[dtype], B, Cc, H, W, patch, pixels.data_ptr(), out.data_ptr(), out.stride(0)))
    return out


def image_normalize(images, rescale, mean=None, std=None, out=None):
    """(B, C, H, W) uint8 or fp32 on the device -> fp32 (x * rescale - mean[c]) / std[c]  (klab_image_normalize)."""
    assert images.is_cuda and images.is_contiguous() and images.dim() == 4 and images.dtype in (torch.uint8, torch.float32)
    B, Cc, H, W = images.shape
    y = torch.empty(B, Cc, H, W, dtype=torch.float32, device=images.device) if out is None else out
    has = mean is not None
    m = (C.c_float * Cc)(*[float(v) for v in (mean if has else [0.0] * Cc)])
    s = (C.c_float * Cc)(*[float(v) for v in (std if has else [1.0] * Cc)])
    L.check(L.lib().klab_image_normalize(_stream(), int(images.dtype == torch.uint8), B, Cc, H * W, images.data_ptr(), float(rescale), C.cast(m, C.c_void_p),
                                         C.cast(s, C.c_void_p), int(has), y.data_ptr()))
    return y


def patch_merge(x, B, res, Cc, scatter=False):
    """gather: x [B*res*res, C] -> [B*(res/2)^2, 4C];  scatter: the inverse."""
    assert x.is_contiguous()
    if scatter:
        out = torch.empty(B * res * res, Cc, dtype=x.dtype, device=x.device)
    else:
        out = torch.empty(B * (res // 2) ** 2, 4 * Cc, dtype=x.dtype, device=x.device)
    L.check(L.lib().klab_patch_merge(_stream(), _DT[x.dtype], B, res, Cc, x.data_ptr(), out.data_ptr(), int(scatter)))
    return out


def ce_fwd(logits, V, labels):
    rows = logits.shape[0]
    dev = logits.device
    lse = torch.empty(rows, dtype=torch.float32, device=dev)
    row_loss = torch.empty(rows, dtype=torch.float32, device=dev)
    stats = torch.empty(2, dtype=torch.float32, device=dev)
    L.check(L.lib().klab_ce_fwd(_stream(), _DT[logits.dtype], rows, V, logits.data_ptr(), logits.stride(0), labels.data_ptr(),
                                lse.data_ptr(), row_loss.data_ptr(), stats.data_ptr(), err_flag(dev).data_ptr()))
    return lse, stats


def ce_bwd(logits, V, ld_pad, labels, lse, stats, gscale):
    rows = logits.shape[0]
    L.check(L.lib().klab_ce_bwd(_stream(), _DT[logits.dtype], rows, V, logits.data_ptr(), logits.stride(0), ld_pad,
                                labels.data_ptr(), lse.data_ptr(), stats.data_ptr(), _p(gscale)))


def lmhead_ce_fwd(h, table, alpha, labels):
    """Fused LM head + cross entropy forward (bf16 tcgen05 path): the logits (alpha * h table^T) are never written.
    Returns (lse [rows] fp32, stats [2] fp32 = {mean loss over non-ignored rows, #non-ignored rows})."""
    rows, d = h.shape
    V = table.shape[0]
    assert h.dtype == torch.bfloat16 and table.dtype == torch.bfloat16 and h.stride(1) == 1 and table.stride(1) == 1
    dev = h.device
    lse = torch.empty(rows, dtype=torch.float32, device=dev)
    stats = torch.empty(2, dtype=torch.float32, device=dev)
    ws = _bytes(L.lib().klab_lmhead_ce_workspace_bytes(rows, V), dev)
    L.check(L.lib().klab_lmhead_ce_fwd(_stream(), rows, V, d, h.data_ptr(), h.stride(0), table.data_ptr(), table.stride(0), alpha,
                                       labels.data_ptr(), lse.data_ptr(), stats.data_ptr(), ws.data_ptr(), err_flag(dev).data_ptr()))
    return lse, stats


def lmhead_ce_bwd_chunk(h, table, alpha, labels, lse, stats, gscale, v0, vc, out):
    """d loss / d logits (times *gscale) of vocabulary columns [v0, v0 + vc), recomputed from h and table, bf16 into out[:, :vc]."""
    rows, d = h.shape
    chunk = table[v0:v0 + vc]
    L.check(L.lib().klab_lmhead_ce_bwd_chunk(_stream(), rows, d, h.data_ptr(), h.stride(0), chunk.data_ptr(), chunk.stride(0), alpha,
                                             labels.data_ptr(), lse.data_ptr(), stats.data_ptr(), _p(gscale), v0, vc, out.data_ptr(),
                                             out.stride(0)))
    return out[:, :vc]


def cast(x, dtype, out=None):
    x = x.contiguous()
    y = torch.empty(x.shape, dtype=dtype, device=x.device) if out is None else out
    L.check(L.lib().klab_cast(_stream(), _DT[x.dtype], _DT[dtype], x.numel(), x.data_ptr(), y.data_ptr()))
    return y


def dropout_apply(x, p, seed, seed_ptr=None):
    x = x.contiguous()
    y = torch.empty_like(x)
    L.check(L.lib().klab_dropout_apply(_stream(), _DT[x.dtype], x.numel(), x.data_ptr(), y.data_ptr(), p, seed, _p(seed_ptr)))
    return y


def seed_advance(counter: torch.Tensor) -> None:
    """Step the device-side dropout counter (uint64 stored in an int64 tensor) once per training step."""
    L.check(L.lib().klab_seed_advance(_stream(), counter.data_ptr()))
