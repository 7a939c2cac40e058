"""Kernel-level parity (B200 only): every C-ABI kernel family against the oracle / plain torch fp32 on the CPU,
on the same seeded inputs.  Tolerances: fp32 path 1e-4 of the tensor's scale, bf16 path 2e-2."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from oracle import swinv2 as osw  # noqa: E402
from oracle import t5 as ot5  # noqa: E402

DTYPES = [torch.float32, torch.bfloat16]


def ops():
    from klab_multimodalmodel_b200 import ops as o
    return o


def L():
    from klab_multimodalmodel_b200 import _lib
    return _lib


def tol(dtype):
    return 1e-4 if dtype == torch.float32 else 2e-2


def close(got, ref, dtype, what="", scale=None):
    got = got.detach().float().cpu()
    ref = ref.detach().float().cpu()
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    s = ref.abs().max().item() if scale is None else scale
    err = (got - ref).abs().max().item()
    assert err <= tol(dtype) * max(s, 1e-6) + 1e-7, f"{what}: max err {err:.3e} vs scale {s:.3e} ({dtype})"


def rnd(*shape, dtype, seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    x = (torch.randn(*shape, generator=g) * scale)
    xq = x.to(dtype)
    return xq.cuda(), xq.float()          # device tensor, exact fp32 copy of what the device sees


# ------------------------------------------------------------------------------------------------ GEMM
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("a_mn,b_mn", [(0, 0), (0, 1), (1, 1), (1, 0)])
@pytest.mark.parametrize("M,N,K", [(128, 64, 64), (200, 136, 96), (520, 1032, 264), (96, 40, 48)])
def test_gemm_layouts(dtype, a_mn, b_mn, M, N, K):
    o = ops()
    A, Ar = rnd(M, K, dtype=dtype, seed=1)
    B, Br = rnd(N, K, dtype=dtype, seed=2)
    a = A.t().contiguous() if a_mn else A
    b = B.t().contiguous() if b_mn else B
    d = o.gemm(a, b, M, N, K, a_mn=bool(a_mn), b_mn=bool(b_mn), out_dtype=torch.float32)
    close(d, Ar @ Br.t(), torch.float32 if dtype == torch.float32 else dtype, "gemm")


@pytest.mark.parametrize("dtype", DTYPES)
def test_gemm_epilogues(dtype):
    o, lib = ops(), L()
    M, N, K = 300, 200, 104
    A, Ar = rnd(M, K, dtype=dtype, seed=1)
    B, Br = rnd(N, K, dtype=dtype, seed=2, scale=0.2)
    bias = torch.randn(N, generator=torch.Generator().manual_seed(3))
    R, Rr = rnd(M, N, dtype=dtype, seed=4)
    base = Ar @ Br.t()
    # bias + gelu with pre-activation copy + residual
    pre = torch.empty(M, N, dtype=dtype, device="cuda")
    d = o.gemm(A, B, M, N, K, bias=bias.cuda(), act=lib.ACT_GELU, aux_out=pre, residual=R)
    close(pre, base + bias, dtype, "aux_out")
    close(d, F.gelu(base + bias) + Rr, dtype, "gelu+res")
    # relu, alpha, fp32 output, accumulate
    acc0 = torch.randn(M, N, generator=torch.Generator().manual_seed(5))
    d2 = acc0.clone().cuda()
    o.gemm(A, B, M, N, K, act=lib.ACT_RELU, alpha=0.5, out=d2, accumulate=True)
    close(d2, torch.relu(0.5 * base) + acc0, dtype, "relu+acc")
    # activation backward epilogues
    H, Hr = rnd(M, N, dtype=dtype, seed=6)
    d3 = o.gemm(A, B, M, N, K, act=lib.ACT_RELU_BWD, aux_in=H)
    close(d3, base * (Hr > 0), dtype, "relu_bwd")
    d4 = o.gemm(A, B, M, N, K, act=lib.ACT_GELU_BWD, aux_in=H)
    x = Hr.clone().requires_grad_(True)
    F.gelu(x).backward(base)
    close(d4, x.grad, dtype, "gelu_bwd")
    # GELU whose derivative is saved by the forward epilogue, and the multiply-only backward epilogue that consumes it
    gp = torch.empty(M, N, dtype=dtype, device="cuda")
    d6 = o.gemm(A, B, M, N, K, bias=bias.cuda(), act=lib.ACT_GELU_SAVE_GRAD, aux_out=gp)
    xg = (base + bias).clone().requires_grad_(True)
    F.gelu(xg).sum().backward()
    close(d6, F.gelu(base + bias), dtype, "gelu (save grad)")
    close(gp, xg.grad, dtype, "saved gelu'")
    d7 = o.gemm(A, B, M, N, K, act=lib.ACT_MUL_AUX, aux_in=H)
    close(d7, base * Hr, dtype, "mul_aux")
    # padded leading dimension (vocab not a multiple of 8)
    d5 = o.gemm(A, B, M, N - 3, K, ldd_pad=N)
    close(d5, base[:, :N - 3], dtype, "ldd_pad")


@pytest.mark.parametrize("M,N,K", [(256, 768, 3072), (40, 136, 2048), (512, 2304, 1536)])
def test_gemm_skinny_split_k_with_epilogue(M, N, K):
    """Single-token decode GEMMs (M = batch): K is split across CTAs and the reduce kernel applies the whole epilogue
    (bias, ReLU, residual, bf16 output).  Same result as the unsplit kernel, to fp32-accumulation accuracy."""
    import ctypes as C
    o, lib = ops(), L()
    A, Ar = rnd(M, K, dtype=torch.bfloat16, seed=1)
    B, Br = rnd(N, K, dtype=torch.bfloat16, seed=2, scale=K ** -0.5)
    R, Rr = rnd(M, N, dtype=torch.bfloat16, seed=3)
    bias = torch.randn(N, generator=torch.Generator().manual_seed(4))
    ref = torch.relu(Ar @ Br.t() + bias) + Rr
    outs = {}
    for name, force in (("auto", (-1, -1, -1)), ("split", (-1, -1, 6)), ("nosplit", (-1, -1, 1))):
        lib.lib().klab_gemm_set_force(*force)
        try:
            outs[name] = o.gemm(A, B, M, N, K, bias=bias.cuda(), act=lib.ACT_RELU, residual=R)
            bn, sp, c2 = C.c_int(0), C.c_int(0), C.c_int(0)
            lib.lib().klab_gemm_last_config(C.byref(bn), C.byref(sp), C.byref(c2))
            if name == "split":
                assert sp.value >= 2, "split-K was not used for a skinny GEMM"
            if name == "nosplit":
                assert sp.value == 1
        finally:
            lib.lib().klab_gemm_set_force(-1, -1, -1)
        close(outs[name], ref, torch.bfloat16, f"skinny gemm ({name})")


def test_gemm_dropout_consistency():
    """The epilogue dropout mask depends only on (seed, element index): the bf16 tcgen05 kernel and the fp32 SIMT kernel
    drop the same elements, and about p of them."""
    o = ops()
    M, N, K = 256, 192, 64
    A, Ar = rnd(M, K, dtype=torch.bfloat16, seed=1)
    B, Br = rnd(N, K, dtype=torch.bfloat16, seed=2)
    d = o.gemm(A, B, M, N, K, out_dtype=torch.float32, dropout_p=0.25, seed=77).cpu()
    d32 = o.gemm(A.float(), B.float(), M, N, K, dropout_p=0.25, seed=77).cpu()
    base = Ar @ Br.t()
    dropped = (d == 0) & (base.abs() > 1e-3)
    assert torch.equal(dropped, (d32 == 0) & (base.abs() > 1e-3))
    frac = dropped.float().mean().item()
    assert 0.22 < frac < 0.28, frac
    keep = ~dropped
    assert torch.allclose(d[keep], base[keep] / 0.75, rtol=1e-2, atol=1e-2)


# ------------------------------------------------------------------------------------------------ norms
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("rows,d", [(37, 64), (260, 768), (5, 1000)])
def test_rmsnorm(dtype, rows, d):
    o = ops()
    X, Xr = rnd(rows, d, dtype=dtype, seed=1)
    DY, DYr = rnd(rows, d, dtype=dtype, seed=2)
    DR, DRr = rnd(rows, d, dtype=dtype, seed=3)
    g = 1 + 0.1 * torch.randn(d, generator=torch.Generator().manual_seed(4))
    y, rstd = o.rmsnorm_fwd(X, g.cuda(), 1e-6)
    xr = Xr.clone().requires_grad_(True)
    gr = g.clone().requires_grad_(True)
    yr = ot5.rms_norm(xr, gr, 1e-6)
    close(y, yr, dtype, "rms fwd")
    yr.backward(DYr)
    dx, dg = o.rmsnorm_bwd(DY, X, g.cuda(), rstd, dres=DR)
    close(dx, xr.grad + DRr, dtype, "rms dx")
    close(dg, gr.grad, dtype, "rms dgamma")


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("rows,d", [(37, 32), (300, 128), (6, 1024)])
def test_layernorm(dtype, rows, d):
    o = ops()
    X, Xr = rnd(rows, d, dtype=dtype, seed=1)
    R, Rr = rnd(rows, d, dtype=dtype, seed=5)
    DY, DYr = rnd(rows, d, dtype=dtype, seed=2)
    gen = torch.Generator().manual_seed(4)
    g = 1 + 0.1 * torch.randn(d, generator=gen)
    b = 0.1 * torch.randn(d, generator=gen)
    y, mean, rstd = o.layernorm_fwd(X, g.cuda(), b.cuda(), 1e-5, residual=R)
    xr, gr, br = Xr.clone().requires_grad_(True), g.clone().requires_grad_(True), b.clone().requires_grad_(True)
    yr = F.layer_norm(xr, (d,), gr, br, 1e-5) + Rr
    close(y, yr, dtype, "ln fwd")
    yr.backward(DYr)
    dx, dg, db = o.layernorm_bwd(DY, X, g.cuda(), mean, rstd)
    close(dx, xr.grad, dtype, "ln dx")
    close(dg, gr.grad, dtype, "ln dgamma")
    close(db, br.grad, dtype, "ln dbeta")
    close(o.colsum(DY), DYr.sum(0), dtype, "colsum")


def test_norm_grouped_output():
    """Writing the two halves of the concat buffer [image tokens; text tokens] (models/model.py:23) in place."""
    o = ops()
    B, n_img, l_src, d = 3, 4, 5, 64
    buf = torch.zeros(B, n_img + l_src, d, device="cuda")
    X, Xr = rnd(B * n_img, d, dtype=torch.float32, seed=1)
    Z, Zr = rnd(B * l_src, d, dtype=torch.float32, seed=2)
    g = torch.ones(d)
    o.layernorm_fwd(X, g.cuda(), torch.zeros(d).cuda(), 1e-5, out=buf, out_rows_per_group=n_img,
                    out_group_stride=(n_img + l_src) * d, save_stats=False)
    o.rmsnorm_fwd(Z, g.cuda(), 1e-6, out=buf[:, n_img:], out_rows_per_group=l_src, out_group_stride=(n_img + l_src) * d,
                  save_stats=False)
    ref = torch.cat([F.layer_norm(Xr, (d,)).view(B, n_img, d), ot5.rms_norm(Zr, g, 1e-6).view(B, l_src, d)], 1)
    close(buf, ref, torch.float32, "concat")


# ------------------------------------------------------------------------------------------------ T5 attention
def _attn_cases(shapes, ps=(0.0, 0.1), multi=False):
    """pytest params (mode, B, H, Lq, Lk, dk, p, multi); the dropout-free cases keep their plain shape ids."""
    out = []
    for shape in shapes:
        for p in ps:
            name = "-".join(map(str, shape)) + (f"-p{p}" if p else "") + ("-multi" if multi else "")
            out.append(pytest.param(*shape, p, multi, id=name))
    return out


# Kernel paths (bf16 needs d_kv = 64 and L <= 256 for tcgen05, everything else runs the generic kernels of t5_attention.cu; fp32
# always does).  Odd Lk makes the dropout element index (bh*Lq + i)*Lk + j change parity from row to row, which reaches the
# odd-base branches that rebuild keep bits one element at a time.
T5_ATTN_SHAPES = [("enc", 2, 3, 13, 13, 64), ("dec", 2, 2, 9, 9, 64), ("cross", 2, 2, 7, 13, 64),
                  ("enc", 1, 2, 81, 81, 16), ("dec", 1, 1, 40, 40, 32),
                  ("enc", 2, 2, 96, 96, 64), ("enc", 1, 2, 176, 176, 64), ("dec", 2, 2, 130, 130, 64),
                  ("cross", 1, 2, 32, 200, 64), ("cross", 2, 1, 150, 96, 64), ("dec", 3, 2, 32, 32, 64),
                  # packed single-tile path: 128 / L problems per tile, partial last tile, both mask kinds
                  ("enc", 9, 2, 32, 32, 64), ("dec", 8, 3, 32, 32, 64), ("dec", 5, 3, 64, 64, 64), ("enc", 2, 2, 64, 64, 64),
                  # backward kernel choice: 32 x 96 (decoder cross-attention of workload 2a) and 96 x 96 take the two-CTA-per-SM
                  # kernel, 128 x 128 / 120 x 100 do not fit twice per SM and take the 512-thread kernel unpacked
                  ("cross", 3, 2, 32, 96, 64), ("enc", 2, 2, 128, 128, 64), ("cross", 3, 2, 120, 100, 64), ("dec", 2, 2, 113, 113, 64),
                  # bf16 generic kernels with L > 256 (odd Lk too); multi-tile tcgen05 kernels with an odd Lk > 128
                  ("enc", 1, 2, 300, 300, 64), ("cross", 2, 1, 24, 301, 64), ("cross", 2, 2, 40, 139, 64)]
# the multi-tile tcgen05 kernels forced at single-tile shapes (KLAB_T5_ATTN_MULTI is read on every call)
T5_ATTN_MULTI_SHAPES = [("enc", 2, 3, 13, 13, 64), ("dec", 5, 3, 64, 64, 64), ("cross", 3, 2, 32, 96, 64), ("dec", 2, 2, 113, 113, 64)]


def t5_attention_reference(QKVr, DOr, table, mode, B, H, Lq, Lk, dk, mask=None):
    """float64 T5 attention (oracle arithmetic, no projections) -> (ctx, lse, dq, dk, dv, dtable | None).  mask: the dropout
    multipliers [B, H, Lq, Lk] (0 or 65536 / thr16) applied to the probabilities before they meet V."""
    dims = ot5.T5Dims(num_heads=H, d_kv=dk)
    inner = H * dk
    QKVd = QKVr.double()
    qr = QKVd[:B * Lq, :inner].clone().requires_grad_(True)
    kr = QKVd[:B * Lk, inner:2 * inner].clone().requires_grad_(True)
    vr = QKVd[:B * Lk, 2 * inner:].clone().requires_grad_(True)
    tr = table.double().clone().requires_grad_(True)
    s = qr.view(B, Lq, H, dk).transpose(1, 2) @ kr.view(B, Lk, H, dk).transpose(1, 2).transpose(-1, -2)
    if mode != "cross":
        s = s + ot5.t5_bias(tr, Lq, Lk, bidirectional=(mode == "enc"), dims=dims)[None]
    if mode == "dec":
        s = s + torch.where(torch.arange(Lk)[None, :] > torch.arange(Lq)[:, None], torch.finfo(torch.float32).min, 0.0).double()
    p = torch.softmax(s, -1)
    if mask is not None:
        p = p * mask
    ref = (p @ vr.view(B, Lk, H, dk).transpose(1, 2)).transpose(1, 2).reshape(B * Lq, inner)
    ref.backward(DOr.double())
    return (ref.detach(), torch.logsumexp(s.detach(), -1), qr.grad, kr.grad, vr.grad,
            tr.grad if mode != "cross" else None)


def t5_attention_case(dtype, mode, B, H, Lq, Lk, dk, p, seed=0, ctr=None, qk_scale=0.5):
    """Runs the kernels' forward and backward on seeded inputs -> (device outputs, host inputs); ctr: the one-element device
    counter added to the dropout seed (as functional.py passes it)."""
    o = ops()
    inner = H * dk
    QKV, QKVr = rnd(B * max(Lq, Lk), 3 * inner, dtype=dtype, seed=1, scale=qk_scale)      # larger scale: more peaked softmax
    q, k, v = QKV[:B * Lq, :inner], QKV[:B * Lk, inner:2 * inner], QKV[:B * Lk, 2 * inner:]
    DO, DOr = rnd(B * Lq, inner, dtype=dtype, seed=2)
    table = 0.5 * torch.randn(32, H, generator=torch.Generator().manual_seed(3))
    has_bias = mode != "cross"
    lut, rz = o.t5_rel_bucket_lut(Lq, Lk, bidirectional=(mode == "enc"), num_buckets=32, max_distance=128)
    kw = dict(bias_table=table.cuda() if has_bias else None, lut=lut.cuda() if has_bias else None, rel_zero=rz, causal=mode == "dec",
              dropout_p=p, seed=seed, seed_ptr=ctr)
    ctx, lse = o.t5_attention_fwd(q, k, v, B, H, Lq, Lk, dk, **kw)
    dQKV = torch.zeros_like(QKV)
    dq, dk_, dv = dQKV[:B * Lq, :inner], dQKV[:B * Lk, inner:2 * inner], dQKV[:B * Lk, 2 * inner:]
    dtab = torch.zeros(32, H, device="cuda")
    o.t5_attention_bwd(q, k, v, ctx, DO, lse, dq, dk_, dv, B, H, Lq, Lk, dk, dbias_table=dtab if has_bias else None, **kw)
    return (ctx, lse, dq, dk_, dv, dtab if has_bias else None), (QKVr, DOr, table)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("mode,B,H,Lq,Lk,dk,p,multi", _attn_cases(T5_ATTN_SHAPES) + _attn_cases(T5_ATTN_MULTI_SHAPES, multi=True))
def test_t5_attention(dtype, mode, B, H, Lq, Lk, dk, p, multi, monkeypatch):
    """Forward (ctx and the un-dropped lse) and backward (dq, dk, dv, bias-table gradient) of every T5 attention kernel path
    against float64.  With p > 0 the reference multiplies the probabilities by the mask `dropout_apply` draws over a
    contiguous [B, H, Lq, Lk] tensor of ones (element (b, h, i, j) at ((b*H + h)*Lq + i)*Lk + j, the index every attention
    kernel hashes), seeded through a device counter."""
    if multi:
        monkeypatch.setenv("KLAB_T5_ATTN_MULTI", "1")
    seed, ctr = 1234, torch.tensor([987654321], dtype=torch.int64, device="cuda")
    got, (QKVr, DOr, table) = t5_attention_case(dtype, mode, B, H, Lq, Lk, dk, p, seed=seed, ctr=ctr)
    mask = ops().dropout_apply(torch.ones(B, H, Lq, Lk, device="cuda"), p, seed, ctr).double().cpu() if p > 0 else None
    ref = t5_attention_reference(QKVr, DOr, table, mode, B, H, Lq, Lk, dk, mask)
    for name, g, r in zip(("t5 attn fwd", "t5 lse", "t5 dq", "t5 dk", "t5 dv", "t5 dbias"), got, ref):
        if r is not None:
            close(g, r, dtype, name)


@pytest.mark.parametrize("mode,B,H,Lk,dk,t", [("self", 5, 3, 20, 64, 0), ("self", 5, 3, 20, 64, 7), ("self", 3, 2, 20, 64, 19), ("cross", 4, 12, 96, 64, 0),
                                              ("cross", 3, 2, 177, 64, 0), ("self", 2, 2, 40, 32, 33), ("cross", 2, 1, 50, 128, 0),
                                              ("cross", 260, 12, 96, 64, 0)])
def test_t5_attention_decode_shape(mode, B, H, Lk, dk, t):
    """K14: one query row per (batch, head) against cached keys / values (the single-token decoder step): the bandwidth-shaped
    kernel.  self: causal with q_offset = t over a [B, T, 3*inner] cache whose rows beyond t hold stale garbage; cross: all keys."""
    o = ops()
    dims = ot5.T5Dims(num_heads=H, d_kv=dk)
    inner = H * dk
    dtype = torch.bfloat16
    cache, cacher = rnd(B * Lk, 3 * inner, dtype=dtype, seed=1, scale=0.5)
    Q, Qr = rnd(B, inner, dtype=dtype, seed=2, scale=0.5)
    k, v = cache[:, inner:2 * inner], cache[:, 2 * inner:]
    table = 0.5 * torch.randn(32, H, generator=torch.Generator().manual_seed(3))
    if mode == "self":
        lut, rz = o.t5_rel_bucket_lut(Lk, Lk, bidirectional=False, num_buckets=32, max_distance=128)
        ctx, lse = o.t5_attention_fwd(Q, k, v, B, H, 1, Lk, dk, bias_table=table.cuda(), lut=lut.cuda(), rel_zero=rz, causal=True, q_offset=t)
        nk = t + 1
    else:
        ctx, lse = o.t5_attention_fwd(Q, k, v, B, H, 1, Lk, dk)
        nk = Lk
    kr = cacher[:, inner:2 * inner].view(B, Lk, H, dk)[:, :nk].transpose(1, 2)
    vr = cacher[:, 2 * inner:].view(B, Lk, H, dk)[:, :nk].transpose(1, 2)
    s = Qr.view(B, 1, H, dk).transpose(1, 2) @ kr.transpose(-1, -2)                       # [B, H, 1, nk]
    if mode == "self":
        s = s + ot5.t5_bias(table, Lk, Lk, bidirectional=False, dims=dims)[None, :, t:t + 1, :nk]
    ref = (torch.softmax(s, -1) @ vr).transpose(1, 2).reshape(B, inner)
    close(ctx, ref, dtype, "t5 decode attn")
    close(lse.view(B, H), torch.logsumexp(s, -1).view(B, H), torch.float32, "t5 decode lse", scale=None)


def test_t5_bucket_lut_matches_oracle():
    o = ops()
    for bidir in (True, False):
        lut, rz = o.t5_rel_bucket_lut(200, 300, bidir, 32, 128)
        rel = torch.arange(-199, 300)
        ref = ot5.relative_position_bucket(rel, bidir, 32, 128)
        assert torch.equal(lut.long(), ref) and rz == 199


# ------------------------------------------------------------------------------------------------ Swin attention
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("B,res,heads,hd,w,shift", [(2, 8, 2, 32, 4, 2), (1, 8, 1, 32, 8, 0), (2, 14, 2, 32, 7, 3), (1, 16, 3, 16, 4, 0),
                                                    (24, 32, 3, 32, 8, 4),      # 576 (head, pair) items: persistent CTAs loop, prefetch, and change head mid-range
                                                    (3, 7, 1, 32, 7, 0),        # odd window count: padded second slot
                                                    (2, 24, 2, 32, 12, 6),      # 12 x 12 windows (384^2 inputs), N = 144: two query passes per window
                                                    (3, 12, 1, 32, 12, 0),      # grid == window: one unshifted 144-token window per image
                                                    (8, 48, 3, 32, 12, 6),      # 384 (head, window) items: CTAs loop over windows and change head
                                                    (1, 18, 2, 32, 9, 4), (2, 20, 1, 32, 10, 5), (1, 22, 2, 32, 11, 5)])   # 81 / 100 / 121 tokens: one pass
def test_swin_attention(dtype, B, res, heads, hd, w, shift):
    o = ops()
    Cc = heads * hd
    n = w * w
    QKV, QKVr = rnd(B * res * res, 3 * Cc, dtype=dtype, seed=1)
    DO, DOr = rnd(B * res * res, Cc, dtype=dtype, seed=2)
    gen = torch.Generator().manual_seed(3)
    sd = {
        "logit_scale": (math.log(10.0) + 0.3 * torch.randn(heads, 1, 1, generator=gen)),
        "continuous_position_bias_mlp.0.weight": torch.randn(512, 2, generator=gen) * 0.7,
        "continuous_position_bias_mlp.0.bias": torch.randn(512, generator=gen) * 0.05,
        "continuous_position_bias_mlp.2.weight": torch.randn(heads, 512, generator=gen) * 0.05,
    }
    sd["logit_scale"][0] = 5.0                                   # exercises the clamp at ln(100)
    sd = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    coords, index = o.swin_tables(w, 0)
    assert torch.equal(index.long(), osw.position_index(w)) and torch.allclose(coords, osw.coords_table(w, 0))
    w1, b1, w2 = (sd["continuous_position_bias_mlp.0.weight"], sd["continuous_position_bias_mlp.0.bias"],
                  sd["continuous_position_bias_mlp.2.weight"])
    bias, hidden, tab = o.swin_cpb_fwd(coords.cuda(), index.cuda(), w1.detach().cuda(), b1.detach().cuda(), w2.detach().cuda(), heads, n)
    bias_ref = osw.cpb_bias(sd, "", w, 0, heads)
    close(bias, bias_ref, torch.float32, "cpb bias")
    ls = sd["logit_scale"].detach().view(-1).cuda()
    q, k, v = QKV[:, :Cc], QKV[:, Cc:2 * Cc], QKV[:, 2 * Cc:]
    ctx, lse = o.swin_attention_fwd(q, k, v, B, res, heads, hd, w, shift, ls, bias)
    # reference: roll -> partition -> cosine attention -> reverse -> roll back (oracle/swinv2.py)
    qkvr = QKVr.clone().requires_grad_(True)
    xs = qkvr.view(B, res, res, 3 * Cc)
    if shift:
        xs = torch.roll(xs, (-shift, -shift), (1, 2))
    win = osw._partition(xs, w)
    bw = win.shape[0]
    qq, kk, vv = [t.reshape(bw, n, heads, hd).transpose(1, 2) for t in win.split(Cc, dim=-1)]
    s = F.normalize(qq, dim=-1) @ F.normalize(kk, dim=-1).transpose(-1, -2)
    s = s * torch.clamp(sd["logit_scale"], max=math.log(100.0)).exp() + bias_ref[None]
    mask = osw.shift_mask(res, res, w, shift)
    if mask is not None:
        nw = mask.shape[0]
        s = (s.view(bw // nw, nw, heads, n, n) + 2 * mask[None, :, None]).view(bw, heads, n, n)
    out = (torch.softmax(s, -1) @ vv).transpose(1, 2).reshape(bw, n, Cc)
    out = osw._reverse(out, w, res, res)
    if shift:
        out = torch.roll(out, (shift, shift), (1, 2))
    ref = out.reshape(B * res * res, Cc)
    close(ctx, ref, dtype, "swin attn fwd")
    ref.backward(DOr)
    dQKV = torch.zeros_like(QKV)
    dbias, dls = o.swin_attention_bwd(q, k, v, ctx, DO, dQKV[:, :Cc], dQKV[:, Cc:2 * Cc], dQKV[:, 2 * Cc:], B, res, heads, hd, w,
                                      shift, ls, bias, lse)
    close(dQKV, qkvr.grad, dtype, "swin dqkv")
    # d(logit_scale) is one scalar per head summed over every window with heavy cancellation: in bf16 the rounding of P and
    # ctx (which feed D_i = dO_i . O_i) shifts it by a few percent; 5e-2 of the largest entry there, 1e-4 in fp32
    ref_dls = sd["logit_scale"].grad.view(-1)
    if dtype == torch.bfloat16:
        close(dls, ref_dls, dtype, "swin dlogit_scale", scale=2.5 * ref_dls.abs().max().item())
    else:
        close(dls, ref_dls, dtype, "swin dlogit_scale")
    dw1, db1, dw2 = o.swin_cpb_bwd(coords.cuda(), index.cuda(), w2.detach().cuda(), hidden, tab, dbias, heads, n)
    slack = 2.0 if dtype == torch.bfloat16 else 1.0         # the bias gradient sums bf16-rounded dS over all windows
    close(dw2, w2.grad, dtype, "cpb dw2", scale=slack * w2.grad.abs().max().item())
    close(dw1, w1.grad, dtype, "cpb dw1", scale=slack * w1.grad.abs().max().item())
    close(db1, b1.grad, dtype, "cpb db1", scale=slack * b1.grad.abs().max().item())


# ------------------------------------------------------------------------------------------------ data movement + CE
@pytest.mark.parametrize("dtype", DTYPES)
def test_embedding_patch_ce(dtype):
    o = ops()
    # embedding with shift_right (labels contain -100) and scatter-add backward
    V, d, B, Lx = 50, 32, 3, 6
    T, Tr = rnd(V, d, dtype=dtype, seed=1)
    labels = torch.randint(2, V, (B, Lx), generator=torch.Generator().manual_seed(2))
    labels[:, -2:] = -100
    dims = ot5.T5Dims(vocab_size=V)
    e = o.embedding_fwd(labels.cuda(), T, shift_right=True)
    ids = ot5.shift_right(labels, dims)
    close(e, Tr[ids].view(B * Lx, d), dtype, "embedding")
    DO, DOr = rnd(B * Lx, d, dtype=dtype, seed=3)
    dT = torch.zeros(V, d, device="cuda")
    o.embedding_bwd(labels.cuda(), DO, dT, shift_right=True)
    ref = torch.zeros(V, d).index_add_(0, ids.view(-1), DOr)
    close(dT, ref, dtype, "embedding bwd")
    # patchify == conv2d(k = s = 4) as a GEMM
    px = torch.randn(2, 3, 16, 24, generator=torch.Generator().manual_seed(4))
    W, Wr = rnd(8, 48, dtype=dtype, seed=5, scale=0.2)
    pm = o.patchify(px.cuda(), 4, dtype)
    y = o.linear_fwd(pm, W, out_dtype=torch.float32)
    ref = F.conv2d(pm.float().cpu().view(2, 4, 6, 3, 4, 4).permute(0, 3, 1, 4, 2, 5).reshape(2, 3, 16, 24), Wr.view(8, 3, 4, 4), stride=4)
    close(y, ref.flatten(2).transpose(1, 2).reshape(-1, 8), dtype, "patch embed")
    assert torch.equal(pm.float().cpu().view(2, 4, 6, 3, 4, 4).permute(0, 3, 1, 4, 2, 5).reshape(2, 3, 16, 24).to(dtype), px.to(dtype))
    # patch merging gather / scatter
    X, Xr = rnd(2 * 6 * 6, 8, dtype=dtype, seed=6)
    g = o.patch_merge(X, 2, 6, 8)
    gg = Xr.view(2, 6, 6, 8)
    ref = torch.cat([gg[:, 0::2, 0::2], gg[:, 1::2, 0::2], gg[:, 0::2, 1::2], gg[:, 1::2, 1::2]], -1).reshape(-1, 32)
    assert torch.equal(g.float().cpu(), ref)
    assert torch.equal(o.patch_merge(g, 2, 6, 8, scatter=True).float().cpu(), Xr)
    # cross entropy with ignore_index
    rows, Vv = B * Lx, 43
    LG, LGr = rnd(rows, 48, dtype=dtype, seed=7, scale=2.0)
    lg = LG[:, :Vv]
    lab = labels.clamp(max=Vv - 1).view(-1)
    lab[labels.view(-1) == -100] = -100
    lse, stats = o.ce_fwd(lg, Vv, lab.cuda())
    lr = LGr[:, :Vv].clone().requires_grad_(True)
    loss = F.cross_entropy(lr, lab, ignore_index=-100)
    close(stats[:1], loss.view(1), dtype, "ce loss")
    loss.backward()
    gs = torch.tensor([0.5], device="cuda")
    o.ce_bwd(lg, Vv, 48, lab.cuda(), lse, stats, gs)
    close(LG[:, :Vv], 0.5 * lr.grad, dtype, "ce bwd")
    assert (LG[:, Vv:] == 0).all()
    o.check_err_flag(LG.device)


@pytest.mark.parametrize("rows,d,ld", [(5000, 512, 512), (4099, 128, 384), (777, 96, 96), (9001, 1536, 1536), (3, 256, 256), (70000, 384, 1152)])
def test_colsum_shapes(rows, d, ld):
    """Bias-gradient column sums: the 16-byte bf16 path (d % 8 == 0, strided rows as in dqkv slices), its scalar fallback and
    the 32-lane finalize, at row counts that exercise several row chunks."""
    o = ops()
    gen = torch.Generator().manual_seed(rows + d)
    full = torch.randn(rows, ld, generator=gen)
    for dtype in (torch.bfloat16, torch.float32):
        X = full.to(dtype).cuda()
        view = X[:, ld - d:]
        ref = view.float().cpu().double().sum(0)
        got = o.colsum(view).cpu().double()
        tol = 2e-5 * math.sqrt(rows) * 4 + 1e-6
        assert (got - ref).abs().max().item() <= tol * max(1.0, ref.abs().max().item()), (dtype, (got - ref).abs().max().item())


def test_fused_adam_refreshes_bf16_operands():
    """The optimizer pass also rewrites the bf16 operand copies the tensor cores read (no cast kernels in a training step):
    after klab Adam the OperandCache entry is fresh and equals bf16(master); after a foreign optimizer (torch.optim.Adam
    bumps the version counters) `get` notices and re-casts."""
    from klab_multimodalmodel_b200 import ops as O
    from klab_multimodalmodel_b200.functional import OperandCache
    from klab_multimodalmodel_b200.optim import Adam
    torch.manual_seed(1)
    ps = [torch.randn(64, 256, device="cuda").requires_grad_() for _ in range(3)] + [torch.randn(40, 256, device="cuda").requires_grad_()]
    cache = OperandCache()
    qkv = cache.get(ps[:3], torch.bfloat16)
    solo = cache.get(ps[3:], torch.bfloat16)
    assert torch.equal(qkv, torch.cat([p.detach() for p in ps[:3]]).bfloat16())
    opt = Adam(ps, lr=1e-2)
    for _ in range(2):
        for p in ps:
            p.grad = torch.randn_like(p)
        v0 = [p._version for p in ps]
        opt.step()
        assert all(p._version > v for p, v in zip(ps, v0))
        n0 = O.launch_count()
        assert cache.get(ps[:3], torch.bfloat16).data_ptr() == qkv.data_ptr() and cache.get(ps[3:], torch.bfloat16).data_ptr() == solo.data_ptr()
        assert O.launch_count() == n0, "operand copies were re-cast although the optimizer refreshed them"
        assert torch.equal(qkv, torch.cat([p.detach() for p in ps[:3]]).bfloat16())
        assert torch.equal(solo, ps[3].detach().bfloat16())
    # a group only partly owned by the optimizer must NOT be marked fresh
    opt2 = Adam(ps[:2], lr=1e-2)
    for p in ps[:2]:
        p.grad = torch.randn_like(p)
    with torch.no_grad():
        ps[2].add_(1.0)
    opt2.step()
    n0 = O.launch_count()
    assert torch.equal(cache.get(ps[:3], torch.bfloat16), torch.cat([p.detach() for p in ps[:3]]).bfloat16())
    assert O.launch_count() > n0
    # foreign optimizer
    topt = torch.optim.Adam(ps, lr=1e-2)
    for p in ps:
        p.grad = torch.randn_like(p)
    topt.step()
    assert torch.equal(cache.get(ps[:3], torch.bfloat16), torch.cat([p.detach() for p in ps[:3]]).bfloat16())


def test_fused_adam_side_stream_only_for_declared_parameters():
    """The update leaves the compute stream only when EVERY parameter of the step was declared by its owner with allow_overlap()
    (MyModel: the trainable transformer, which forward() reads after wait_pending_updates()).  Anything else -- a plain tensor
    list, an optimizer over model.parameters() -- runs on the current stream like torch.optim.Adam; either way the values a
    consumer sees after wait_pending_updates() are the updated ones."""
    from klab_multimodalmodel_b200 import optim as KO
    torch.manual_seed(3)
    ps = [torch.randn(300, 257, device="cuda").requires_grad_() for _ in range(4)]
    ref = [p.detach().clone().requires_grad_() for p in ps]
    oa, ob = KO.Adam(ps, lr=1e-2), torch.optim.Adam(ref, lr=1e-2)

    def one_step():
        for p, r in zip(ps, ref):
            p.grad = torch.randn_like(p)
            r.grad = p.grad.clone()
        oa.step(); ob.step()

    KO._DONE.clear()
    one_step()
    assert not KO._DONE, "an optimizer over undeclared parameters must stay on the current stream"
    KO.allow_overlap(ps[:3])
    one_step()
    assert not KO._DONE, "one undeclared parameter in the step keeps it on the current stream"
    KO.allow_overlap(ps)
    one_step()
    if KO.OVERLAP:
        assert KO._DONE, "all parameters declared: the update runs on the side stream"
    one_step()                                                # a second update while the first is still pending: ordered
    KO.wait_pending_updates(ps[0].device)
    assert not KO._DONE
    for p, r in zip(ps, ref):                                 # read on the compute stream after the wait
        assert (p.detach() - r.detach()).abs().max().item() <= 1e-6 * max(1.0, r.detach().abs().max().item())
    for p in ps:
        KO._OVERLAP_SAFE.pop(id(p), None)


def test_fused_adam_matches_torch_adam():
    """N1: klab Adam == torch.optim.Adam (train.py:28) over several steps, odd sizes, an unaligned view, weight decay and an
    LR scheduler; state_dict keys are torch's.  Both are fp32 implementations of the same recurrence, so the yardstick is a
    float64 evaluation of it: our distance to it may not exceed torch's (x4, plus one fp32 ulp of slack)."""
    from klab_multimodalmodel_b200.optim import Adam
    torch.manual_seed(0)
    flat = torch.randn(70000, device="cuda")
    shapes = [(1024, 1024), (33, 7), (1,), (16385,), (513, 129)]
    ps_a = [torch.randn(s, device="cuda").requires_grad_() for s in shapes] + [flat[1:50001].detach().clone().requires_grad_()]
    ps_b = [p.detach().clone().requires_grad_() for p in ps_a]
    for wd in (0.0, 0.01):
        lr0, b1, b2, eps = 3e-3, 0.9, 0.98, 1e-8
        oa = Adam(ps_a, lr=lr0, betas=(b1, b2), eps=eps, weight_decay=wd)
        ob = torch.optim.Adam(ps_b, lr=lr0, betas=(b1, b2), eps=eps, weight_decay=wd)
        sa = torch.optim.lr_scheduler.CosineAnnealingLR(oa, T_max=10)
        sb = torch.optim.lr_scheduler.CosineAnnealingLR(ob, T_max=10)
        ex = [dict(p=p.detach().double(), m=torch.zeros_like(p, dtype=torch.float64), v=torch.zeros_like(p, dtype=torch.float64), t=0)
              for p in ps_b]
        for step in range(6):
            lr = oa.param_groups[0]["lr"]
            assert abs(lr - ob.param_groups[0]["lr"]) < 1e-12
            for k, (pa, pb) in enumerate(zip(ps_a, ps_b)):
                g = torch.randn_like(pa) * (10.0 ** (step - 3))
                pa.grad = g.clone()
                pb.grad = g.clone()
                if step == 3 and k == 1:           # a parameter without a gradient is skipped (and its step count does not advance)
                    pa.grad = None
                    pb.grad = None
                    continue
                e = ex[k]
                e["t"] += 1
                gd = g.double() + wd * e["p"]
                e["m"] = b1 * e["m"] + (1 - b1) * gd
                e["v"] = b2 * e["v"] + (1 - b2) * gd * gd
                e["p"] = e["p"] - (lr / (1 - b1 ** e["t"])) * e["m"] / (e["v"].sqrt() / (1 - b2 ** e["t"]) ** 0.5 + eps)
            oa.step(); ob.step(); sa.step(); sb.step()
        for k, (pa, pb) in enumerate(zip(ps_a, ps_b)):
            for name, xa, xb, xe in (("param", pa, pb, ex[k]["p"]), ("exp_avg", oa.state[pa]["exp_avg"], ob.state[pb]["exp_avg"], ex[k]["m"]),
                                     ("exp_avg_sq", oa.state[pa]["exp_avg_sq"], ob.state[pb]["exp_avg_sq"], ex[k]["v"])):
                ea = (xa.detach().double() - xe).abs().max().item()
                eb = (xb.detach().double() - xe).abs().max().item()
                ulp = 1.2e-7 * xe.abs().max().item()
                assert ea <= 4.0 * eb + ulp, f"tensor {k} {name}: klab error {ea:.3e} vs torch error {eb:.3e} against float64"
        sd = oa.state_dict()
        assert set(sd["state"][0]) == {"step", "exp_avg", "exp_avg_sq"}
        ob2 = torch.optim.Adam(ps_b, lr=1e-3)
        ob2.load_state_dict(sd)                 # torch's Adam accepts our state (python-int step counts included)
        for pa, pb in zip(ps_a, ps_b):          # keep the two trajectories identical for the next round
            pb.data.copy_(pa.data)


@pytest.mark.parametrize("rows,V,d", [(300, 1000, 128), (64, 32128, 256), (2048, 520, 64)])
def test_fused_lmhead_cross_entropy(rows, V, d):
    """K10 hot path: LM head fused with the cross entropy (logits never written) against fp32 torch on the same bf16 operands:
    lse / mean loss with ignore_index, an out-of-range label raises, and the chunked d loss / d logits."""
    from klab_multimodalmodel_b200 import ops as o
    torch.manual_seed(rows + V)
    h = (torch.randn(rows, d, device="cuda") * 2.0).bfloat16()
    E = (torch.randn(V, d, device="cuda") * 1.5).bfloat16()
    labels = torch.randint(0, V, (rows,), device="cuda")
    labels[::7] = -100
    labels[1] = V - 1
    labels[2] = 0
    alpha = d ** -0.5
    ref_logits = (h.float() @ E.float().t()) * alpha
    ref_lse = torch.logsumexp(ref_logits, dim=-1)
    ref_loss = torch.nn.functional.cross_entropy(ref_logits, labels, ignore_index=-100)
    lse, stats = o.lmhead_ce_fwd(h, E, alpha, labels)
    o.check_err_flag(h.device)
    torch.testing.assert_close(lse, ref_lse, rtol=1e-4, atol=1e-3)
    assert abs(stats[0].item() - ref_loss.item()) <= 1e-4 * abs(ref_loss.item()) + 1e-4
    assert stats[1].item() == float((labels != -100).sum().item())
    # backward, chunked: (softmax - onehot) * g / n_valid, zero rows for ignored labels
    g = torch.tensor([0.37], device="cuda")
    ref_d = torch.softmax(ref_logits, dim=-1)
    valid = labels != -100
    ref_d[valid, labels[valid]] -= 1.0
    ref_d = ref_d * (0.37 / valid.sum().item())
    ref_d[~valid] = 0.0
    chunk = 512 if V > 512 else 264
    scratch = torch.empty(rows, chunk, dtype=torch.bfloat16, device="cuda")
    for v0 in range(0, V, chunk):
        vc = min(chunk, V - v0)
        dl = o.lmhead_ce_bwd_chunk(h, E, alpha, labels, lse, stats, g, v0, vc, scratch)
        ref = ref_d[:, v0:v0 + vc]
        err = (dl.float() - ref).abs().max().item()
        assert err <= 1e-2 * ref.abs().max().item() + 1e-7, (v0, err)
    bad = labels.clone()
    bad[5] = V + 3
    o.lmhead_ce_fwd(h, E, alpha, bad)
    with pytest.raises(IndexError):
        o.check_err_flag(h.device)


# ------------------------------------------------------------------------------------------------ dynamic work distribution
def test_dynamic_work_distribution_matches_static():
    """klab_set_dynamic_sched(1) (what the data-parallel reducer arms): the persistent GEMM and T5-attention kernels claim
    work items from a per-launch counter.  Results must be bit-identical to the static stride (the atomically reduced bias
    gradient: to fp32 rounding), also when a launch has many
    more items than CTAs, uses split-K, is replayed from a CUDA graph (the last CTA re-arms the counter) and when far more
    launches than counter slots have been issued."""
    o, lib = ops(), L()
    dev = "cuda"

    def run_all():
        outs = []
        for (M, N, K, a_mn, b_mn, od) in [(4096, 2048, 256, False, False, torch.bfloat16), (1000, 520, 136, False, True, torch.bfloat16),
                                          (512, 384, 4096, True, True, torch.float32), (20000, 128, 64, False, False, torch.bfloat16)]:
            A, _ = rnd(K if a_mn else M, M if a_mn else K, dtype=torch.bfloat16, seed=M)
            B, _ = rnd(K if b_mn else N, N if b_mn else K, dtype=torch.bfloat16, seed=N)
            outs.append(o.gemm(A, B, M, N, K, a_mn=a_mn, b_mn=b_mn, out_dtype=od))
        Bt, H, Lq, dk = 40, 8, 48, 64                      # 320 problems > 148 CTAs (48: not packed into shared tiles)
        QKV, _ = rnd(Bt * Lq, 3 * H * dk, dtype=torch.bfloat16, seed=7, scale=0.5)
        q, k, v = QKV[:, :H * dk], QKV[:, H * dk:2 * H * dk], QKV[:, 2 * H * dk:]
        table = (0.5 * torch.randn(32, H, generator=torch.Generator().manual_seed(3))).cuda()
        lut, rz = o.t5_rel_bucket_lut(Lq, Lq, bidirectional=False, num_buckets=32, max_distance=128)
        kw = dict(bias_table=table, lut=lut.cuda(), rel_zero=rz, causal=True)
        ctx, lse = o.t5_attention_fwd(q, k, v, Bt, H, Lq, Lq, dk, **kw)
        DO, _ = rnd(Bt * Lq, H * dk, dtype=torch.bfloat16, seed=8)
        dQKV = torch.zeros_like(QKV)
        dtab = torch.zeros_like(table)
        o.t5_attention_bwd(q, k, v, ctx, DO, lse, dQKV[:, :H * dk], dQKV[:, H * dk:2 * H * dk], dQKV[:, 2 * H * dk:], Bt, H, Lq, Lq, dk,
                           dbias_table=dtab, **kw)
        return outs + [ctx, lse, dQKV, dtab]

    static = run_all()
    # the CTA-pair GEMM (tcgen05.mma.cta_group::2) with its leader-claims-for-the-pair queue: pinned, static vs dynamic
    def run_pairs():
        import ctypes as C
        outs = []
        lib.lib().klab_gemm_set_force(1, -1, -1)
        try:
            for (M, N, K, a_mn, b_mn, od) in [(6144, 1024, 1024, False, True, torch.bfloat16), (4096, 2048, 256, False, False, torch.bfloat16),
                                              (1024, 4096, 6144, True, True, torch.float32), (300, 520, 136, False, False, torch.bfloat16),
                                              (40000, 256, 128, False, False, torch.bfloat16)]:
                A, _ = rnd(K if a_mn else M, M if a_mn else K, dtype=torch.bfloat16, seed=M + 1)
                B, _ = rnd(K if b_mn else N, N if b_mn else K, dtype=torch.bfloat16, seed=N + 1)
                outs.append(o.gemm(A, B, M, N, K, a_mn=a_mn, b_mn=b_mn, out_dtype=od))
                c2 = C.c_int(0)
                lib.lib().klab_gemm_last_config(None, None, C.byref(c2))
                assert c2.value == 1, "the CTA-pair kernel was not used"
        finally:
            lib.lib().klab_gemm_set_force(-1, -1, -1)
        return outs

    static_pairs = run_pairs()
    lib.lib().klab_set_dynamic_sched(1)
    try:
        dyn = run_all()
        for s_, d_ in zip(static[:-1], dyn[:-1]):
            assert torch.equal(s_, d_)
        # the relative-position bias gradient is summed with shared-memory float atomics (diagonal sums of several warps meet in
        # one slot; the order is not fixed), like the scatter-add of the reference's embedding backward: equal to fp32 rounding
        assert (static[-1] - dyn[-1]).abs().max().item() <= 1e-5 * max(1.0, static[-1].abs().max().item())
        for rep in range(3):                               # counters re-armed by the last pair: repeated launches agree
            for s_, d_ in zip(static_pairs, run_pairs()):
                assert torch.equal(s_, d_)
        # graph replay: the counters must be back at zero after every launch
        A, _ = rnd(2048, 512, dtype=torch.bfloat16, seed=11)
        B, _ = rnd(1024, 512, dtype=torch.bfloat16, seed=12)
        D = torch.empty(2048, 1024, dtype=torch.bfloat16, device=dev)
        o.gemm(A, B, 2048, 1024, 512, out=D)
        ref = D.clone()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(3):
                o.gemm(A, B, 2048, 1024, 512, out=D)
        for _ in range(4):
            D.zero_()
            g.replay()
            assert torch.equal(D, ref)
        # slot reuse: more launches than the 8192 counter slots
        small_a, _ = rnd(256, 64, dtype=torch.bfloat16, seed=13)
        small_b, _ = rnd(128, 64, dtype=torch.bfloat16, seed=14)
        first = o.gemm(small_a, small_b, 256, 128, 64)
        for _ in range(9000):
            last = o.gemm(small_a, small_b, 256, 128, 64)
        assert torch.equal(first, last)
    finally:
        lib.lib().klab_set_dynamic_sched(0)


# ------------------------------------------------------------------------------------------------ N2: host input path
@pytest.mark.parametrize("in_dtype", [torch.uint8, torch.float32])
@pytest.mark.parametrize("shape", [(3, 3, 256, 256), (2, 3, 7, 9)])
def test_image_normalize_matches_host_processor(in_dtype, shape):
    """N2: rescale (1/255) + ImageNet normalise on the device (klab_image_normalize) against the host arithmetic it replaces
    (/root/reference/train.py:55, transformers ViTImageProcessor): bit-exact with the numpy restatement of the slow processor,
    within 2e-6 of the installed transformers processor itself (its torch path fuses the two steps)."""
    from klab_multimodalmodel_b200.data import GpuImageProcessor
    g = torch.Generator().manual_seed(5)
    x = torch.randint(0, 256, shape, generator=g).to(torch.uint8) if in_dtype == torch.uint8 else torch.rand(shape, generator=g)
    proc = GpuImageProcessor.from_pretrained("microsoft/swinv2-base-patch4-window8-256", size=shape[-2:])
    batch = proc(x, return_tensors="pt").to("cuda")
    got = batch["pixel_values"]
    assert got.dtype == torch.float32 and got.is_cuda and got.shape == x.shape
    ref = proc.preprocess_on_host(x)
    assert torch.equal(got.cpu(), ref), (got.cpu() - ref).abs().max()
    # a second batch through the same pinned staging pair, channels-last list input
    y = [im.permute(1, 2, 0) for im in x] if shape[-1] != 3 else None
    if y is not None:
        again = proc(y).to(torch.device("cuda"))["pixel_values"]
        assert torch.equal(again.cpu(), ref)
    try:
        from transformers import ViTImageProcessor
    except ImportError:
        return
    hf = ViTImageProcessor(do_resize=False, image_mean=list(proc.image_mean), image_std=list(proc.image_std))
    want = hf(x, return_tensors="pt")["pixel_values"]
    assert (got.cpu() - want).abs().max().item() <= 2e-6 * max(1.0, want.abs().max().item())


def test_device_prefetcher_overlaps_and_preserves_order():
    """N2: batches come out in order, already on the device and normalised, one step of look-ahead on a side stream."""
    from klab_multimodalmodel_b200.data import DevicePrefetcher, GpuImageProcessor
    proc = GpuImageProcessor(size=(16, 16))
    g = torch.Generator().manual_seed(9)
    host = [(torch.rand(4, 3, 16, 16, generator=g).pin_memory(), torch.randint(0, 100, (4, 5), generator=g).pin_memory()) for _ in range(5)]
    dev = torch.device("cuda", 0)

    def transform(b):
        px, ids = b
        return proc(px).to(dev), {"input_ids": ids.to(dev, non_blocking=True)}

    seen = 0
    for i, (images, src) in enumerate(DevicePrefetcher(host, dev, transform)):
        torch.cuda.current_stream().synchronize()
        assert torch.equal(images["pixel_values"].cpu(), proc.preprocess_on_host(host[i][0]))
        assert torch.equal(src["input_ids"].cpu(), host[i][1])
        seen += 1
    assert seen == 5


def test_greedy_step_argmax_ties_and_finished_rows():
    """K14: ids[b, t] = argmax of the fp32 logits row (LOWEST index on ties, as torch.argmax), pad for finished rows, EOS finishes a row."""
    lib = L()
    B, V = 7, 32128
    g = torch.Generator().manual_seed(11)
    logits = torch.randn(B, V, generator=g)
    logits[0, 5] = logits[0, 31000] = 9.0                     # tie: first index wins
    logits[1, 1] = 20.0                                       # EOS
    logits[2, V - 1] = 15.0
    want = logits.argmax(-1)
    ids = torch.zeros(B, 4, dtype=torch.int64, device="cuda")
    alive = torch.ones(B, dtype=torch.int32, device="cuda")
    alive[3] = 0
    lg = logits.cuda()
    lib.check(lib.lib().klab_greedy_step(torch.cuda.current_stream().cuda_stream, B, V, lg.data_ptr(), lg.stride(0), ids.data_ptr(),
                                         ids.stride(0), 2, alive.data_ptr(), 0, 1))
    got = ids[:, 2].cpu()
    want[3] = 0
    assert torch.equal(got, want) and got[0].item() == 5
    assert alive.cpu().tolist() == [1, 0, 1, 0, 1, 1, 1]
    # unaligned / odd vocabulary: scalar path
    lg2 = logits[:, :1001].contiguous().cuda()
    lib.check(lib.lib().klab_greedy_step(torch.cuda.current_stream().cuda_stream, B, 1001, lg2.data_ptr(), lg2.stride(0), ids.data_ptr(),
                                         ids.stride(0), 3, alive.data_ptr(), 0, 1))
    w2 = logits[:, :1001].argmax(-1)
    w2[1] = 0
    w2[3] = 0
    assert torch.equal(ids[:, 3].cpu(), w2)
