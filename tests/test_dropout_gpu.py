"""Training-mode dropout, kernel level (B200 only).  Every dropout mask of the library is a pure function of (seed + device
counter, element index), and `klab_dropout_apply` exposes that generator: applied to a tensor of ones it yields the mask of any
site.  These tests use it as the mask oracle -- the hash is never restated -- and prove that each kernel applies exactly that
mask, then check the arithmetic around it in float64 (T5 attention: tests/test_kernels_gpu.py::test_t5_attention)."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from tests.test_kernels_gpu import close, ops, rnd, t5_attention_case, t5_attention_reference, tol  # noqa: E402
from oracle import t5 as ot5  # noqa: E402

DTYPES = [torch.float32, torch.bfloat16]
P = 0.1


def L():
    from klab_multimodalmodel_b200 import _lib
    return _lib


def ctr_of(value):
    return torch.tensor([value], dtype=torch.int64, device="cuda")


def mask_of(shape, p, seed, ctr=None):
    """The multipliers (0 or 65536 / thr16) a dropout site with this seed applies to a contiguous tensor of `shape`."""
    return ops().dropout_apply(torch.ones(*shape, device="cuda"), p, seed, ctr).double().cpu()


# ------------------------------------------------------------------------------------------------ dropout_apply, seed_advance
@pytest.mark.parametrize("dtype", DTYPES)
def test_dropout_apply_multiplier_fraction_and_odd_length(dtype):
    """klab_dropout_apply: survivors are scaled by exactly 65536 / thr16 (not 1 / (1 - p)), the kept fraction is within 4 sigma of
    thr16 / 65536, an odd length takes the last element through the scalar tail, and x * mask is rounded once to the dtype."""
    o = ops()
    for p in (0.1, 0.25, 0.5):
        thr16 = min(65536, max(1, int((1.0 - p) * 65536.0 + 0.5)))
        mult = np.float32(65536.0) / np.float32(thr16)
        n = (1 << 20) + 1
        m = o.dropout_apply(torch.ones(n, device="cuda"), p, 99, None).cpu()
        kept = m != 0
        assert torch.all(m[kept] == torch.tensor(float(mult))), (p, m[kept].unique())
        q = thr16 / 65536.0
        frac = kept.double().mean().item()
        assert abs(frac - q) <= 4 * (q * (1 - q) / n) ** 0.5, (p, frac, q)
        for n_odd in (1, 3, 1001, 4097):
            x, xr = rnd(n_odd, dtype=dtype, seed=n_odd)
            y = o.dropout_apply(x, p, 7, ctr_of(11)).cpu()
            mk = mask_of((n_odd,), p, 7, ctr_of(11)).float()
            assert torch.equal(y, (xr * mk).to(dtype)), (p, n_odd)


def test_seed_advance_is_the_64_bit_lcg():
    """klab_seed_advance steps the device counter by c <- c * 6364136223846793005 + 1442695040888963407 (mod 2^64), stored in an
    int64 tensor; the counter is added to every site's seed, so masks after a step differ."""
    o = ops()
    for start in (0, 1, 123456789, (1 << 62) + 5, -3):
        c = ctr_of(start)
        want = start % (1 << 64)
        for _ in range(3):
            o.seed_advance(c)
            want = (want * 6364136223846793005 + 1442695040888963407) % (1 << 64)
            got = int(c.item()) % (1 << 64)
            assert got == want, (start, got, want)
    c = ctr_of(5)
    before = mask_of((4096,), P, 3, c)
    o.seed_advance(c)
    assert not torch.equal(before, mask_of((4096,), P, 3, c))


# ------------------------------------------------------------------------------------------------ T5 attention
# one entry per kernel path (tcgen05 kernels: bf16 with d_kv = 64, L <= 256):
PROBE_CASES = [
    ("enc", 1, 2, 81, 81, 16, False),      # generic kernels (d_kv != 64), odd Lk; fp32: SIMT kernels at every shape
    ("enc", 1, 2, 300, 300, 64, False),    # generic kernels, L > 256
    ("enc", 9, 2, 32, 32, 64, False),      # single-tile tcgen05 forward (and backward), packed 4 per tile, B = 9 not a multiple of 4
    ("dec", 5, 3, 64, 64, 64, False),      # packed 2 per tile, causal, odd B; backward: 512-thread kernel packed
    ("enc", 2, 3, 13, 13, 64, False),      # single-tile forward unpacked, odd Lk; backward: two-CTA kernel
    ("cross", 3, 2, 32, 96, 64, False),    # two-CTA backward (decoder cross-attention of the benchmark)
    ("dec", 2, 2, 113, 113, 64, False),    # 512-thread single-tile backward, odd Lk
    ("cross", 3, 2, 120, 100, 64, False),  # 512-thread single-tile backward
    ("cross", 2, 2, 40, 139, 64, False),   # multi-tile forward and backward, odd Lk > 128
    ("enc", 1, 2, 176, 176, 64, False),    # multi-tile, 128 < L <= 256
    ("enc", 2, 3, 13, 13, 64, True),       # multi-tile kernels forced at single-tile shapes (KLAB_T5_ATTN_MULTI=1)
    ("dec", 5, 3, 64, 64, 64, True),
]
PROBE_IDS = ["-".join(map(str, c[:6])) + ("-multi" if c[6] else "") for c in PROBE_CASES]


def probe_keep_mask(dtype, mode, B, H, Lq, Lk, dk, p, seed, ctr):
    """The forward kernel's own keep mask [B, H, Lq, Lk]: q = k = 0 and no bias make P uniform over the visible keys; V is one-hot
    (key j of chunk c writes column j - c*d_kv), so out[b, i, h, j - c*d_kv] > 0 iff element (b, h, i, j) was kept."""
    o = ops()
    inner = H * dk
    q = torch.zeros(B * Lq, inner, dtype=dtype, device="cuda")
    k = torch.zeros(B * Lk, inner, dtype=dtype, device="cuda")
    keep = torch.zeros(B, H, Lq, Lk, dtype=torch.bool)
    for c0 in range(0, Lk, dk):
        n = min(dk, Lk - c0)
        v = torch.zeros(B, Lk, H, dk, dtype=dtype, device="cuda")
        j = torch.arange(c0, c0 + n)
        v[:, j, :, j - c0] = 1.0
        ctx, _ = o.t5_attention_fwd(q, k, v.view(B * Lk, inner), B, H, Lq, Lk, dk, causal=mode == "dec", dropout_p=p, seed=seed,
                                    seed_ptr=ctr)
        out = ctx.float().cpu().view(B, Lq, H, dk).permute(0, 2, 1, 3)              # [B, H, Lq, d_kv]
        keep[..., c0:c0 + n] = out[..., :n] > 0
    return keep


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("mode,B,H,Lq,Lk,dk,multi", PROBE_CASES, ids=PROBE_IDS)
def test_t5_attention_forward_mask_is_dropout_apply(dtype, mode, B, H, Lq, Lk, dk, multi, monkeypatch):
    """Bit-exact keep mask of every T5 attention forward path (fp32 SIMT t5_attn_fwd_kernel, bf16 generic kernel, tcgen05
    single-tile packed / unpacked and multi-tile kernels): it equals dropout_apply over a contiguous [B, H, Lq, Lk] tensor of
    ones, and the device counter is added to the seed (seed 1000 + counter 234 draws the mask of seed 1234 without one)."""
    if multi:
        monkeypatch.setenv("KLAB_T5_ATTN_MULTI", "1")
    keep = probe_keep_mask(dtype, mode, B, H, Lq, Lk, dk, P, 1000, ctr_of(234))
    want = mask_of((B, H, Lq, Lk), P, 1234) > 0
    if mode == "dec":                                         # masked keys have P = 0: only the visible ones carry the mask
        vis = torch.arange(Lk)[None, :] <= torch.arange(Lq)[:, None]
        want = want & vis
    bad = (keep != want).nonzero()
    assert bad.shape[0] == 0, f"{bad.shape[0]} elements differ from dropout_apply, first (b, h, i, j) {bad[:4].tolist()}"


def _manual_attention_grads(QKVr, DOr, table, mode, B, H, Lq, Lk, dk, mask, variant=None):
    """float64 attention with hand-written backward -> (ctx, dq, dk, dv); `variant` applies one plausible kernel bug."""
    dims = ot5.T5Dims(num_heads=H, d_kv=dk)
    inner = H * dk
    X = QKVr.double()
    q = X[:B * Lq, :inner].view(B, Lq, H, dk).transpose(1, 2)
    k = X[:B * Lk, inner:2 * inner].view(B, Lk, H, dk).transpose(1, 2)
    v = X[:B * Lk, 2 * inner:].view(B, Lk, H, dk).transpose(1, 2)
    dO = DOr.double().view(B, Lq, H, dk).transpose(1, 2)
    s = q @ k.transpose(-1, -2)
    if mode != "cross":
        s = s + ot5.t5_bias(table.double(), Lq, Lk, bidirectional=(mode == "enc"), dims=dims)[None]
    if mode == "dec":
        s = s + torch.where(torch.arange(Lk)[None, :] > torch.arange(Lq)[:, None], torch.finfo(torch.float32).min, 0.0).double()
    P_ = torch.softmax(s, -1)
    if variant == "no mask":
        mask = torch.ones_like(mask)
    elif variant == "neighbouring (b, h)":
        mask = mask.reshape(B * H, Lq, Lk).roll(1, 0).view(B, H, Lq, Lk)
    Pd = P_ * mask
    ctx = (Pd @ v).transpose(1, 2).reshape(B * Lq, inner)
    dPd = dO @ v.transpose(-1, -2)
    dP = dPd * mask
    D = (Pd * dPd).sum(-1, keepdim=True)
    if variant == "D from un-dropped P":
        D = (P_ * dPd).sum(-1, keepdim=True)
    dS = P_ * (dP - D)
    if variant == "dS = 0 where dropped":
        dS = torch.where(mask > 0, dS, torch.zeros_like(dS))
    dq = (dS @ k).transpose(1, 2).reshape(B * Lq, inner)
    dk_ = (dS.transpose(-1, -2) @ q).transpose(1, 2).reshape(B * Lk, inner)
    dv = (Pd.transpose(-1, -2) @ dO).transpose(1, 2).reshape(B * Lk, inner)
    return ctx, dq, dk_, dv


def _rel_err(got, ref):
    return ((got.double() - ref.double()).abs().max() / ref.double().abs().max().clamp_min(1e-6)).item()


@pytest.mark.parametrize("mode,B,H,Lq,Lk,dk,multi", PROBE_CASES, ids=PROBE_IDS)
def test_t5_attention_bf16_tolerance_sees_dropout_bugs(mode, B, H, Lq, Lk, dk, multi, monkeypatch):
    """The 2e-2 bf16 bound of the attention parity test can see wrong dropout: for each bf16 path the float64 reference evaluated
    under a plausible bug (no mask, the mask of the neighbouring (b, h), the mask shifted by one key, dS = 0 on dropped elements,
    D_i from the un-dropped P) lies at least 3x the bound away from the correct one on some output, at an input scale (peaked
    softmax) chosen until it does -- and the kernels stay within the bound there."""
    if multi:
        monkeypatch.setenv("KLAB_T5_ATTN_MULTI", "1")
    dtype, seed, ctr = torch.bfloat16, 1000, ctr_of(234)
    mask = mask_of((B, H, Lq, Lk), P, seed, ctr)
    # element e of the shifted mask is element e + 1 of the true one
    shifted = ops().dropout_apply(torch.ones(B * H * Lq * Lk + 1, device="cuda"), P, seed, ctr).double().cpu()[1:].view(B, H, Lq, Lk)
    variants = ("no mask", "neighbouring (b, h)", "shifted by one key", "dS = 0 where dropped", "D from un-dropped P")
    names = ("ctx", "dq", "dk", "dv")
    for scale in (0.5, 1.0, 2.0):
        got, (QKVr, DOr, table) = t5_attention_case(dtype, mode, B, H, Lq, Lk, dk, P, seed=seed, ctr=ctr, qk_scale=scale)
        ref = _manual_attention_grads(QKVr, DOr, table, mode, B, H, Lq, Lk, dk, mask)
        auto = t5_attention_reference(QKVr, DOr, table, mode, B, H, Lq, Lk, dk, mask)
        for name, a, b in zip(names, ref, (auto[0], auto[2], auto[3], auto[4])):
            assert _rel_err(a, b) < 1e-10, f"hand-written backward disagrees with autograd on {name}"
        seen = {}
        for var in variants:
            if var == "shifted by one key":
                alt = _manual_attention_grads(QKVr, DOr, table, mode, B, H, Lq, Lk, dk, shifted)
            else:
                alt = _manual_attention_grads(QKVr, DOr, table, mode, B, H, Lq, Lk, dk, mask, variant=var)
            seen[var] = max(_rel_err(x, r) for x, r in zip(alt, ref))
        if min(seen.values()) >= 3 * tol(dtype):
            break
    assert min(seen.values()) >= 3 * tol(dtype), f"input scale {scale}: a bug variant hides inside the bound: {seen}"
    for name, g, r in zip(names, (got[0], got[2], got[3], got[4]), ref):
        close(g, r, dtype, f"{name} (q/k scale {scale})")


# ------------------------------------------------------------------------------------------------ rmsnorm_bwd(drop=...)
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("rows,d", [(37, 512), (20, 768), (9, 1024),        # vector kernel with the fused dropout output
                                    (37, 64), (5, 1000), (6, 2048)])        # two-pass fallback: rmsnorm_bwd, then dropout_apply
def test_rmsnorm_bwd_dropout(dtype, rows, d):
    """rmsnorm_bwd(drop=(p, seed, counter)) -- the fused "dropout of the consumer's output gradient" of functional.py's T5 block
    backward: dx and dgamma against float64, and dx_drop is dropout_apply(dx) bit for bit (mask of a contiguous [rows, d]
    tensor, applied to the stored dx), so its zeros are exactly those of the mask."""
    o = ops()
    X, Xr = rnd(rows, d, dtype=dtype, seed=1)
    DY, DYr = rnd(rows, d, dtype=dtype, seed=2)
    DR, DRr = rnd(rows, d, dtype=dtype, seed=3)
    g = 1 + 0.1 * torch.randn(d, generator=torch.Generator().manual_seed(4))
    _, rstd = o.rmsnorm_fwd(X, g.cuda(), 1e-6)
    ctr = ctr_of(555)
    dx, dg, dxd = o.rmsnorm_bwd(DY, X, g.cuda(), rstd, dres=DR, drop=(P, 77, ctr))
    xr = Xr.double().clone().requires_grad_(True)
    gr = g.double().clone().requires_grad_(True)
    ot5.rms_norm(xr, gr, 1e-6).backward(DYr.double())
    ref_dx = xr.grad + DRr.double()
    mask = mask_of((rows, d), P, 77, ctr)
    close(dx, ref_dx, dtype, "rms dx")
    close(dg, gr.grad, dtype, "rms dgamma")
    close(dxd, ref_dx * mask, dtype, "rms dx_drop")
    assert torch.equal(dxd.cpu(), o.dropout_apply(dx, P, 77, ctr).cpu()), "dx_drop is not dropout_apply(dx)"
    dxc = dx.float().cpu()
    assert torch.equal((dxd.float().cpu() == 0) & (dxc != 0), (mask == 0) & (dxc != 0))


# ------------------------------------------------------------------------------------------------ GEMM epilogue dropout
def _gemm_kernels():
    return [("fp32 SIMT", torch.float32, None), ("bf16 one CTA", torch.bfloat16, 0), ("bf16 CTA pair", torch.bfloat16, 1)]


@pytest.mark.parametrize("kernel", [k[0] for k in _gemm_kernels()])
def test_gemm_epilogue_dropout(kernel):
    """The GEMM epilogue's dropout (act, then mask, then residual) on the fp32 SIMT kernel and on the bf16 tcgen05 kernel pinned
    to one CTA and to a CTA pair: forward with ReLU (the T5 FFN's first GEMM), dgrad with ACT_RELU_BWD + dropout (its
    backward), dropout + residual (the sub-layer outputs) and a padded leading dimension with an odd N (row bases of both
    parities).  The mask is dropout_apply over a contiguous [M, N] tensor of ones: zero pattern exact, values against float64."""
    _, dtype, cta2 = next(k for k in _gemm_kernels() if k[0] == kernel)
    o, lib = ops(), L()
    M, N, K = 300, 520, 136
    A, Ar = rnd(M, K, dtype=dtype, seed=1)
    Bw, Br = rnd(N, K, dtype=dtype, seed=2, scale=K ** -0.5)
    R, Rr = rnd(M, N, dtype=dtype, seed=3)
    Hs, Hr = rnd(M, N, dtype=dtype, seed=4)
    ctr = ctr_of(42)
    base = Ar.double() @ Br.double().t()
    if cta2 is not None:
        lib.lib().klab_gemm_set_force(cta2, -1, -1)
    try:
        outs = {}

        def run(name, *args, **kw):
            outs[name] = o.gemm(*args, dropout_p=P, seed=kw.pop("seed"), seed_ptr=ctr, **kw)
            if cta2 is not None:
                c2 = C.c_int(-1)
                lib.lib().klab_gemm_last_config(None, None, C.byref(c2))
                assert c2.value == cta2, (name, c2.value)

        run("relu", A, Bw, M, N, K, act=lib.ACT_RELU, seed=10)
        run("residual", A, Bw, M, N, K, residual=R, seed=11)
        run("ldd_pad", A, Bw, M, N - 3, K, ldd_pad=N, act=lib.ACT_RELU, seed=12)
        DYd, DYr = rnd(M, N, dtype=dtype, seed=5)                       # dgrad dx[M, K] = relu'(h) * (dy w) * mask
        Wd, Wr = rnd(N, K, dtype=dtype, seed=6, scale=N ** -0.5)
        Hk, Hkr = rnd(M, K, dtype=dtype, seed=7)
        run("relu_bwd", DYd, Wd, M, K, N, b_mn=True, act=lib.ACT_RELU_BWD, aux_in=Hk, seed=13)      # = linear_dgrad(dy, w)
    finally:
        lib.lib().klab_gemm_set_force(-1, -1, -1)
    refs = {
        "relu": (torch.relu(base) * mask_of((M, N), P, 10, ctr), torch.relu(base)),
        "residual": (base * mask_of((M, N), P, 11, ctr) + Rr.double(), None),
        "ldd_pad": (torch.relu(base[:, :N - 3]) * mask_of((M, N - 3), P, 12, ctr), torch.relu(base[:, :N - 3])),
    }
    pre = DYr.double() @ Wr.double()                                  # [M, N] x [N, K]
    refs["relu_bwd"] = (pre * (Hkr.double() > 0) * mask_of((M, K), P, 13, ctr), pre * (Hkr.double() > 0))
    for name, (ref, premask) in refs.items():
        got = outs[name]
        close(got, ref, dtype, f"{kernel} {name}")
        if premask is not None:
            g = got.float().cpu()
            live = premask.abs() > 1e-3 * premask.abs().max()         # elements the activation kept, clear of rounding to zero
            assert torch.equal((g == 0) & live, (ref == 0) & live), f"{kernel} {name}: zero pattern differs from the mask"
