"""Block-level forward/backward schedules of the caption step, as torch.autograd.Functions over the C-ABI kernels.

Granularity is one autograd node per transformer block (plus embed / merge / loss nodes) so that gradients of a block's
parameters become ready as soon as its backward finishes: DistributedDataParallel's bucket all-reduce
(/root/reference/train.py:26,62) then overlaps the rest of the backward pass (SURVEY.md section 8e).  The kernel sequence
of each block is captured into a CUDA graph per shape signature (graphs.py), so the host issues ~170 graph launches per
step instead of ~4000 kernel launches.

Every arithmetic step below is a kernel of libklab_b200.so (ops.py); torch supplies memory, streams and the
autograd graph only.  Citations: HF/ = site-packages/transformers 5.5.0.
"""
from __future__ import annotations

import math
import os
import weakref

import torch

from . import _lib as L
from . import ops as O
from .graphs import POOL


# ------------------------------------------------------------------------------------------------
# operand cache: fp32 master weights -> (concatenated) operands in the compute dtype
# ------------------------------------------------------------------------------------------------
# parameter id -> [(weakref to the owning OperandCache, entry key, first row, rows)]: where the compute-dtype copies of a parameter live.  The fused optimizer
# (optim.py) writes the bf16 copy in the same pass that updates the fp32 master and then marks the entry fresh, so a
# training step contains no cast kernels at all.
_PARAM_SLOTS: dict = {}


def operand_slots(p):
    """[(entry, view of the operand rows that hold `p`)] for every cached compute-dtype copy of parameter `p`."""
    out, live = [], []
    for ref, key, r0, r in _PARAM_SLOTS.get(id(p), ()):
        cache = ref()
        e = cache._store.get(key) if cache is not None else None
        if e is None:
            continue                                          # the cache (model) is gone or was cleared: drop the stale slot
        live.append((ref, key, r0, r))
        if e[4][e[5].index(id(p))] is p and e[1].device == p.device:
            out.append((e, e[1][r0:r0 + r]))
    if id(p) in _PARAM_SLOTS:
        _PARAM_SLOTS[id(p)] = live
    return out


def mark_operands_fresh(entries):
    """Called by the optimizer after it rewrote EVERY parameter of each entry (fp32 master and compute-dtype copy alike)."""
    for e in entries:
        e[0] = OperandCache._version(e[4])


class OperandCache:
    """Keeps, per group of parameters, one contiguous [sum(N_i), K] operand in the compute dtype (bf16 copies for the
    tensor cores; q|k|v weights concatenated so one GEMM produces all three).  The buffer of a group never moves, so CUDA
    graphs can bake its address.  `get` refreshes a stale entry eagerly (a parameter's version counter or address changed,
    e.g. after a foreign optimizer's step or load_state_dict); `peek` returns the buffer as is (captured regions and backward
    reuse what `get` validated before the region was launched).  entry = [version, buffer, rows, k, params, param ids]."""

    def __init__(self):
        self._store: dict = {}

    @staticmethod
    def _direct(params, dtype):
        return len(params) == 1 and params[0].dtype == dtype and params[0].dim() == 2

    def _entry(self, params, dtype):
        key = tuple(id(p) for p in params) + (dtype,)
        e = self._store.get(key)
        if e is not None and e[1].device != params[0].device:
            e = None
        if e is None:
            k = params[0][0].numel() if params[0].dim() > 1 else params[0].numel()
            rows = [p.numel() // k for p in params]
            buf = torch.empty(sum(rows), k, dtype=dtype, device=params[0].device)
            e = self._store[key] = [None, buf, rows, k, list(params), [id(p) for p in params]]
            r0, ref = 0, weakref.ref(self)
            for p, r in zip(params, rows):
                _PARAM_SLOTS.setdefault(id(p), []).append((ref, key, r0, r))
                r0 += r
        return e

    @staticmethod
    def _version(params):
        return tuple(p._version for p in params) + tuple(p.data_ptr() for p in params)

    def _convert(self, e, params, dtype):
        buf, rows, k = e[1], e[2], e[3]
        r0 = 0
        for p, r in zip(params, rows):
            O.cast(p.detach().reshape(r, k), dtype, out=buf[r0:r0 + r])
            r0 += r
        e[0] = self._version(params)

    def get(self, params, dtype) -> torch.Tensor:
        if self._direct(params, dtype):
            return params[0].detach()
        e = self._entry(params, dtype)
        if e[0] != self._version(params):
            self._convert(e, params, dtype)
        return e[1]

    def peek(self, params, dtype) -> torch.Tensor:
        if self._direct(params, dtype):
            return params[0].detach()
        return self._entry(params, dtype)[1]

    def clear(self):
        self._store.clear()


def cat_vec(vecs, device) -> torch.Tensor:
    """Concatenate fp32 bias vectors (None -> zeros) with the copy kernel."""
    n = sum(v[1] for v in vecs)
    out = torch.zeros(n, dtype=torch.float32, device=device)
    o = 0
    for t, sz in vecs:
        if t is not None:
            O.cast(t.detach(), torch.float32, out=out[o:o + sz])
        o += sz
    return out


class Ctx:
    """Static description of one block at one shape signature (created once and cached by the owning module, so its
    identity doubles as the CUDA-graph key).  `busy` is set while a captured forward's activations await their backward."""

    def __init__(self, **kw):
        self.busy = False
        self.gen = 0                                # generation of the forward whose static activations are live
        self.__dict__.update(kw)


class _Token:
    """Clears Ctx.busy when the autograd node that owns it dies without having run backward.  Only the token of the LATEST
    captured forward may do so: the previous step's autograd node (kept alive by the caller's `loss` variable) usually dies
    after the next forward has already claimed the Ctx, and must not release it under that forward's pending backward."""

    def __init__(self, c):
        self.c = c
        c.gen += 1
        self.gen = c.gen

    def release(self):
        if self.c.gen == self.gen:
            self.c.busy = False

    def __del__(self):
        self.release()


class _StepToken:
    """Counts training forwards whose backward has not run yet.  While one is outstanding the device-side dropout counter
    must not advance (the pending backward regenerates its masks from it)."""
    outstanding = 0

    def __init__(self):
        self.live = True
        _StepToken.outstanding += 1

    def release(self):
        if self.live:
            self.live = False
            _StepToken.outstanding -= 1

    def __del__(self):
        self.release()


def pending_backward() -> bool:
    return _StepToken.outstanding > 0


_OUTER_GRAD = [True]


def apply_fn(fn_cls, *args):
    """fn_cls.apply(*args), remembering the caller's grad mode: inside Function.forward autograd is always disabled, so the
    decision "keep activations for backward?" has to be taken from the outside (frozen sub-models run under no_grad)."""
    _OUTER_GRAD[0] = torch.is_grad_enabled()
    return fn_cls.apply(*args)


def _needs_grad(tensors) -> bool:
    return _OUTER_GRAD[0] and any(t is not None and t.requires_grad for t in tensors)


# Data parallelism: gradient all-reduces run on NCCL's stream DURING BACKWARD only (reducer.py waits for them at the end of
# backward), so only backward kernels share the GPU with a collective.  While a backward function runs, the library is told to
# distribute GEMM / T5-attention work dynamically and to keep `reserve` SMs out of the statically partitioned Swin kernels;
# forward kernels keep the full machine, the static stride and the CTA-pair GEMM.  (CUDA graphs bake the choice at capture.)
DP_BACKWARD = {"on": False, "reserve": 0}


def _backward_phase(fn):
    def wrapped(ctx, *grads):
        if not DP_BACKWARD["on"]:
            return fn(ctx, *grads)
        lib = L.lib()
        lib.klab_set_dynamic_sched(1)
        lib.klab_set_sm_reserve(DP_BACKWARD["reserve"])
        try:
            return fn(ctx, *grads)
        finally:
            lib.klab_set_dynamic_sched(0)
            lib.klab_set_sm_reserve(0)
    wrapped.__name__ = fn.__name__
    wrapped.__doc__ = fn.__doc__
    return wrapped


ACCUMULATE_IN_PLACE = os.environ.get("KLAB_GRAD_ACCUMULATE_IN_PLACE", "1") != "0"


def _grad_outputs(outs, graphed):
    """Gradients handed back to autograd.  A captured region returns the SAME static tensors on every replay, and its tuple
    keeps a reference to them, so AccumulateGrad (which only adopts a gradient nobody else holds) would clone every parameter
    gradient every step -- ~3 GB of device copies for T5-large.  Fresh aliases of the static storage are adopted as .grad
    without a copy; `_detach_aliased_grads` moves an accumulated value out of the way before the next replay overwrites it."""
    if not graphed:
        return tuple(outs)
    return tuple(o.detach() if torch.is_tensor(o) else o for o in outs)


def _detach_aliased_grads(params):
    """Gradient accumulation: if a parameter's .grad still IS the static gradient buffer of a captured backward region, the
    replay about to run would overwrite it -- move the accumulated value out first."""
    for p in params:
        g = p.grad
        if g is not None and POOL.owns(g):
            p.grad = g.clone()


# ------------------------------------------------------------------------------------------------
# weight-gradient side stream
# ------------------------------------------------------------------------------------------------
class _Side:
    """Weight (and bias) gradients hang off the backward critical path: nothing inside a block consumes them.  They are issued
    on a second stream -- inside a captured region that becomes a parallel branch of the CUDA graph -- so they fill the SMs
    that the latency-bound chain of small dgrad GEMMs / attention / norm kernels leaves idle (the persistent GEMM hands out its
    tiles dynamically, so two GEMMs share the machine gracefully).  All split-K GEMMs of a step are weight gradients and
    therefore serialise on this one stream, which is what their shared fp32 workspace requires (gemm_tc.cu).
    Inputs of a side-stream kernel are kept alive until the join (the caching allocator knows only the allocating stream).
    KLAB_WGRAD_STREAM=0 issues everything on one stream."""
    enabled = os.environ.get("KLAB_WGRAD_STREAM", "1") != "0"
    streams: dict = {}
    keep: list = []
    dirty = False

    @classmethod
    def run(cls, fn, *tensors, **kw):
        if not cls.enabled or not tensors[0].is_cuda:
            return fn(*tensors, **kw)
        main = torch.cuda.current_stream()
        side = cls.streams.get(main.device)
        if side is None:
            side = cls.streams[main.device] = torch.cuda.Stream(main.device)
        side.wait_stream(main)                     # everything issued so far (the operands) happens-before the side kernel
        with torch.cuda.stream(side):
            out = fn(*tensors, **kw)
        cls.keep.extend(tensors)
        cls.dirty = True
        return out

    @classmethod
    def join(cls):
        if cls.dirty:
            main = torch.cuda.current_stream()
            main.wait_stream(cls.streams[main.device])
            cls.keep.clear()
            cls.dirty = False


def _flat_grads(shapes, device):
    """One fp32 buffer for all parameter gradients of a block (segments 32-byte aligned) and a view per parameter: the data-parallel
    reducer then all-reduces ONE large tensor per block instead of a dozen small ones (NCCL's per-operation latency, not its
    bandwidth, bounds a grouped all-reduce over ~1 000 separate tensors)."""
    sizes = [(math.prod(s_) + 7) // 8 * 8 for s_ in shapes]
    flat = torch.empty(sum(sizes), dtype=torch.float32, device=device)
    views, o = [], 0
    for s_, n in zip(shapes, sizes):
        views.append(flat[o:o + math.prod(s_)].view(s_))
        o += n
    return flat, views


def _publish_flat(params, flat, ok):
    """Tell the reducer (reducer.GradReducer._on_grad) that the gradients about to be adopted by `params` are slices of `flat`.
    ok = every parameter's .grad is None right now, i.e. autograd will adopt the slices themselves (no `grad += slice`)."""
    group = {"left": len(params), "flat": flat} if ok and flat is not None else None
    for p in params:
        p._klab_flat = group


def _wgrad(dy, x, **kw):
    return _Side.run(O.linear_wgrad, dy, x, **kw)


def _colsum(dy):
    return _Side.run(O.colsum, dy)


# ------------------------------------------------------------------------------------------------
# T5 block  (HF/models/t5/modeling_t5.py: T5LayerSelfAttention :356-377, T5LayerCrossAttention :387-408,
#            T5LayerFF :135-150, T5Attention :253-344)
# dropout sites of block `c` use seeds c.seed + {0..5} plus the device-side step counter c.seed_ptr
# ------------------------------------------------------------------------------------------------
def _t5_attn_fwd(c, n, kv_src, wq_or_qkv, wkv, wo, resid, table, lut, rz, causal, Lq, Lk, seed, kvbuf=None):
    """n: normed input [B*Lq, d]; returns (h_out, qkv, kvbuf, ctx, lse) with h_out = resid + dropout(attn(n) Wo^T).
    Cross-attention: `kvbuf` = k|v projection of the encoder output, possibly still in flight on the side stream."""
    H, dk = c.H, c.dk
    inner = H * dk
    qkv = O.linear_fwd(n, wq_or_qkv)
    if kv_src is None:                                   # self-attention: one GEMM for q|k|v
        q, k, v = qkv[:, :inner], qkv[:, inner:2 * inner], qkv[:, 2 * inner:]
        kvbuf = None
    else:                                                # cross-attention: q from n, k|v from the encoder output
        q = qkv
        if kvbuf is None:
            kvbuf = O.linear_fwd(kv_src, wkv)
        else:
            _Side.join()
        k, v = kvbuf[:, :inner], kvbuf[:, inner:]
    ctxt, lse = O.t5_attention_fwd(q, k, v, c.B, H, Lq, Lk, dk, bias_table=table, lut=lut, rel_zero=rz,
                                   num_buckets=c.num_buckets, causal=causal, dropout_p=c.p, seed=seed, seed_ptr=c.seed_ptr)
    h = O.linear_fwd(ctxt, wo, residual=resid, dropout_p=c.p, seed=seed + 1, seed_ptr=c.seed_ptr)
    return h, qkv, kvbuf, ctxt, lse


def _t5_attn_bwd(c, dh, n, kv_src, wq_or_qkv, wkv, wo, qkv, kvbuf, ctxt, lse, table, lut, rz, causal, Lq, Lk, seed, dtable, dh_dropped=None,
                 g_wq=None, g_wkv=None, g_wo=None):
    """dh: gradient of the attention layer's output (residual part handled by the caller); dh_dropped: the same with this
    layer's output-dropout mask already applied (fused into the norm backward that produced dh).
    Returns dn, dkv_src (or None), dWq(kv), dWkv (or None), dWo."""
    H, dk = c.H, c.dk
    inner = H * dk
    if dh_dropped is not None:
        dh = dh_dropped
    elif c.p > 0.0:                                      # dropout on the o-projection output (:375 / :406)
        dh = O.dropout_apply(dh, c.p, seed + 1, c.seed_ptr)
    dctx = O.linear_dgrad(dh, wo)
    dwo = _wgrad(dh, ctxt, out=g_wo)
    dqkv = torch.empty_like(qkv)
    if kv_src is None:
        q, k, v = qkv[:, :inner], qkv[:, inner:2 * inner], qkv[:, 2 * inner:]
        dq, dk_, dv = dqkv[:, :inner], dqkv[:, inner:2 * inner], dqkv[:, 2 * inner:]
        dkvbuf = None
    else:
        q, k, v = qkv, kvbuf[:, :inner], kvbuf[:, inner:]
        dkvbuf = torch.empty_like(kvbuf)
        dq, dk_, dv = dqkv, dkvbuf[:, :inner], dkvbuf[:, inner:]
    O.t5_attention_bwd(q, k, v, ctxt, dctx, lse, dq, dk_, dv, c.B, H, Lq, Lk, dk, bias_table=table, lut=lut, rel_zero=rz,
                       num_buckets=c.num_buckets, causal=causal, dbias_table=dtable, dropout_p=c.p, seed=seed, seed_ptr=c.seed_ptr)
    dn = O.linear_dgrad(dqkv, wq_or_qkv)
    dwq = _wgrad(dqkv, n, out=g_wq)
    if kv_src is None:
        return dn, None, dwq, None, dwo
    dkv_src = _Side.run(O.linear_dgrad, dkvbuf, wkv)    # gradient w.r.t. the encoder output: consumed after the block
    dwkv = _wgrad(dkvbuf, kv_src, out=g_wkv)
    return dn, dkv_src, dwq, dwkv, dwo


def _t5_ff_fwd(c, x, ln_w, wi, wo, seed):
    """-> (out, n, rstd, f) or, gated, (out, n, rstd, f, u).  wi: the [wi] or [wi_0; wi_1] operand."""
    n, rstd = O.rmsnorm_fwd(x, ln_w, c.eps)
    if c.gated:                                          # T5DenseGatedActDense (:106-132): one GEMM for both projections
        u = O.linear_fwd(n, wi)
        f = O.geglu_fwd(u, c.p, seed, c.seed_ptr)
    else:
        f = O.linear_fwd(n, wi, act=L.ACT_RELU, dropout_p=c.p, seed=seed, seed_ptr=c.seed_ptr)
    out = O.linear_fwd(f, wo, residual=x, dropout_p=c.p, seed=seed + 1, seed_ptr=c.seed_ptr)
    return (out, n, rstd, f, u) if c.gated else (out, n, rstd, f)


def _t5_ff_bwd(c, dout, x, ln_w, wi, wo, n, rstd, f, seed, next_seed, g_ln=None, g_wi=None, g_wo=None, u=None):
    """next_seed: dropout seed of the sub-layer that consumes dx (its output-dropout mask is applied in the same pass).
    u: the saved [a | b] of the gated FFN.  -> dx, dropout(dx) or None, dln, dwi, dwo"""
    dy = O.dropout_apply(dout, c.p, seed + 1, c.seed_ptr) if c.p > 0.0 else dout
    if c.gated:
        dh = O.linear_dgrad(dy, wo)
        df = O.geglu_bwd(dh, u, c.p, seed, c.seed_ptr)   # [d a | d b]: one dgrad and one wgrad GEMM against [wi_0; wi_1]
    else:
        df = O.linear_dgrad(dy, wo, act=L.ACT_RELU_BWD, aux_in=f, dropout_p=c.p, seed=seed, seed_ptr=c.seed_ptr)
    dwo = _wgrad(dy, f, out=g_wo)
    dn = O.linear_dgrad(df, wi)
    dwi = _wgrad(df, n, out=g_wi)
    if c.p > 0.0:
        dx, dln, dxd = O.rmsnorm_bwd(dn, x, ln_w, rstd, dres=dout, drop=(c.p, next_seed + 1, c.seed_ptr), dgamma_out=g_ln)
    else:
        (dx, dln), dxd = O.rmsnorm_bwd(dn, x, ln_w, rstd, dres=dout, dgamma_out=g_ln), None
    return dx, dxd, dln, dwi, dwo


def _t5_operands(c, params, cd, mode):
    """(wqkv, w_o, w_i, w_ff[, w_cq, w_ckv, w_co]) in the compute dtype; mode in {"get", "peek"}.  Gated: w_i = [wi_0; wi_1]."""
    f = getattr(c.cache, mode)
    if c.is_decoder:
        ln0, q, k, v, o, ln1, cq, ck, cv, co, ln2, *wi, wo = params
        return f([q, k, v], cd), f([o], cd), f(wi, cd), f([wo], cd), f([cq], cd), f([ck, cv], cd), f([co], cd)
    ln0, q, k, v, o, ln1, *wi, wo = params
    return f([q, k, v], cd), f([o], cd), f(wi, cd), f([wo], cd)


def _t5_block_fwd_body(x, enc_out, c, save, table, *params):
    """-> (out,) or (out, n0, rstd0, qkv, ctx, lse, h1, [n1, rstd1, qc, kvbuf, ctx2, lse2, h2,] n2, rstd2, f[, u]); u: gated FFN"""
    cd = x.dtype
    dec = c.is_decoder
    ws = _t5_operands(c, params, cd, "peek")
    seed = c.seed
    if dec:
        ln0, ln1, ln2 = params[0], params[5], params[10]
        wqkv, w_o, w_i, w_ff, w_cq, w_ckv, w_co = ws
    else:
        ln0, ln1 = params[0], params[5]
        wqkv, w_o, w_i, w_ff = ws
    # the k|v projection of the encoder output does not depend on this block's input: side stream, joined before cross-attention
    kv_pre = _Side.run(O.linear_fwd, enc_out, w_ckv) if dec else None
    n0, rstd0 = O.rmsnorm_fwd(x, ln0, c.eps)
    h1, qkv, _, ctxt, lse = _t5_attn_fwd(c, n0, None, wqkv, None, w_o, x, table, c.lut, c.rz, dec, c.L, c.L, seed)
    if dec:
        n1, rstd1 = O.rmsnorm_fwd(h1, ln1, c.eps)
        h2, qc, kvbuf, ctx2, lse2 = _t5_attn_fwd(c, n1, enc_out, w_cq, w_ckv, w_co, h1, None, None, 0, False, c.L, c.Le, seed + 2,
                                                 kvbuf=kv_pre)
        out, *ff = _t5_ff_fwd(c, h2, ln2, w_i, w_ff, seed + 4)
        return (out, n0, rstd0, qkv, ctxt, lse, h1, n1, rstd1, qc, kvbuf, ctx2, lse2, h2, *ff) if save else (out,)
    out, *ff = _t5_ff_fwd(c, h1, ln1, w_i, w_ff, seed + 4)
    return (out, n0, rstd0, qkv, ctxt, lse, h1, *ff) if save else (out,)


def _t5_block_bwd_body(dout, x, enc_out, *rest):
    """rest = saved activations (forward order) then consts (c, table, *params)
    -> (dx, denc | None, dtable | None, *param grads, flat): every parameter gradient is a slice of `flat` (see _flat_grads)"""
    n_acts = 16 if enc_out is not None else 9
    if not isinstance(rest[n_acts], Ctx):                # the gated FFN saves u as well
        n_acts += 1
    acts, (c, table, *params) = rest[:n_acts], rest[n_acts:]
    u = acts[n_acts - 1] if c.gated else None
    cd = x.dtype
    dec = c.is_decoder
    ws = _t5_operands(c, params, cd, "peek")
    seed = c.seed
    inner = c.H * c.dk
    d = x.shape[1]
    dtable = torch.zeros_like(table) if table is not None else None
    denc = None
    if dec:
        n0, rstd0, qkv, ctxt, lse, h1, n1, rstd1, qc, kvbuf, ctx2, lse2, h2, n2, rstd2, f = acts[:16]
        ln0, ln1, ln2 = params[0], params[5], params[10]
        wqkv, w_o, w_i, w_ff, w_cq, w_ckv, w_co = ws
        flat, (g_ln0, g_qkv, g_o, g_ln1, g_cq, g_ckv, g_co, g_ln2, g_wi, g_ff) = _flat_grads(
            [(d,), (3 * inner, d), (d, inner), (d,), (inner, d), (2 * inner, d), (d, inner), (d,), tuple(w_i.shape), tuple(w_ff.shape)], x.device)
        dh2, dh2d, dln2, dwi, dwo_ff = _t5_ff_bwd(c, dout, h2, ln2, w_i, w_ff, n2, rstd2, f, seed + 4, seed + 2, g_ln=g_ln2, g_wi=g_wi, g_wo=g_ff,
                                                  u=u)
        dn1, denc, dwcq, dwckv, dwco = _t5_attn_bwd(c, dh2, n1, enc_out, w_cq, w_ckv, w_co, qc, kvbuf, ctx2, lse2, None, None, 0,
                                                    False, c.L, c.Le, seed + 2, None, dh_dropped=dh2d, g_wq=g_cq, g_wkv=g_ckv, g_wo=g_co)
        if c.p > 0.0:                                    # + the self-attention layer's output-dropout mask for its backward
            dh1, dln1, dh1d = O.rmsnorm_bwd(dn1, h1, ln1, rstd1, dres=dh2, drop=(c.p, seed + 1, c.seed_ptr), dgamma_out=g_ln1)
        else:
            (dh1, dln1), dh1d = O.rmsnorm_bwd(dn1, h1, ln1, rstd1, dres=dh2, dgamma_out=g_ln1), None
    else:
        n0, rstd0, qkv, ctxt, lse, h1, n2, rstd2, f = acts[:9]
        ln0, ln1 = params[0], params[5]
        wqkv, w_o, w_i, w_ff = ws
        flat, (g_ln0, g_qkv, g_o, g_ln1, g_wi, g_ff) = _flat_grads(
            [(d,), (3 * inner, d), (d, inner), (d,), tuple(w_i.shape), tuple(w_ff.shape)], x.device)
        dh1, dh1d, dln1, dwi, dwo_ff = _t5_ff_bwd(c, dout, h1, ln1, w_i, w_ff, n2, rstd2, f, seed + 4, seed, g_ln=g_ln1, g_wi=g_wi, g_wo=g_ff,
                                                  u=u)
    dn0, _, dwqkv, _, dwo = _t5_attn_bwd(c, dh1, n0, None, wqkv, None, w_o, qkv, None, ctxt, lse, table, c.lut, c.rz, dec,
                                         c.L, c.L, seed, dtable, dh_dropped=dh1d, g_wq=g_qkv, g_wo=g_o)
    dx, dln0 = O.rmsnorm_bwd(dn0, x, ln0, rstd0, dres=dh1, dgamma_out=g_ln0)
    _Side.join()
    gq, gk, gv = dwqkv[:inner], dwqkv[inner:2 * inner], dwqkv[2 * inner:]
    gwi = (dwi[:dwi.shape[0] // 2], dwi[dwi.shape[0] // 2:]) if c.gated else (dwi,)      # gated: wi_0 | wi_1
    if dec:
        grads = (dln0, gq, gk, gv, dwo, dln1, dwcq, dwckv[:inner], dwckv[inner:], dwco, dln2, *gwi, dwo_ff)
    else:
        grads = (dln0, gq, gk, gv, dwo, dln1, *gwi, dwo_ff)
    return (dx, denc, dtable) + grads + (flat,)


class T5BlockFn(torch.autograd.Function):
    """One T5Block.  inputs: (c, x, enc_out | None, bias_table | None, *params)
    params (encoder): ln0, q, k, v, o, ln1, wi, wo
    params (decoder): ln0, q, k, v, o, ln1, cq, ck, cv, co, ln2, wi, wo
    (gated FFN: wi_0, wi_1 in place of wi)"""

    @staticmethod
    def forward(ctx, c, x, enc_out, table, *params):
        save = _needs_grad((x, enc_out, table) + tuple(params))
        _t5_operands(c, params, x.dtype, "get")             # stale compute-dtype copies are refreshed eagerly, outside any graph
        x = x.contiguous()
        outs, graphed = POOL.run(("t5f", id(c), save), _t5_block_fwd_body, (x, enc_out), (c, save, table) + tuple(params),
                                 allow_graph=not c.busy)
        if save:
            ctx.c = c
            ctx.graphed = graphed
            ctx.save_for_backward(x, enc_out, table, *params)
            ctx.acts = outs[1:]
            if graphed:
                c.busy = True
                ctx.token = _Token(c)
        return outs[0]

    @staticmethod
    @_backward_phase
    def backward(ctx, dout):
        c = ctx.c
        x, enc_out, table, *params = ctx.saved_tensors
        acts, ctx.acts = ctx.acts, None
        if ctx.graphed:
            _detach_aliased_grads(params if table is None else params + [table])
        outs, graphed = POOL.run(("t5b", id(c)), _t5_block_bwd_body, (dout.contiguous(), x, enc_out) + tuple(acts),
                                 (c, table) + tuple(params), allow_graph=ctx.graphed)
        tok, ctx.token = getattr(ctx, "token", None), None
        if tok is not None:
            tok.release()
        _publish_flat(params, outs[-1], all(p.grad is None for p in params))
        return (None,) + _grad_outputs(outs[:-1], graphed)


# ------------------------------------------------------------------------------------------------
# stand-alone norms (stack outputs) and the concat of [image tokens; text tokens]
# ------------------------------------------------------------------------------------------------
class RMSNormFn(torch.autograd.Function):
    """T5Stack.final_layer_norm (HF/models/t5/modeling_t5.py:767)."""

    @staticmethod
    def forward(ctx, x, w, eps):
        y, rstd = O.rmsnorm_fwd(x, w, eps)
        if _needs_grad((x, w)):
            ctx.save_for_backward(x, w, rstd)
        return y

    @staticmethod
    @_backward_phase
    def backward(ctx, dy):
        x, w, rstd = ctx.saved_tensors
        dx, dw = O.rmsnorm_bwd(dy.contiguous(), x, w, rstd)
        return dx, dw, None


class DropoutFn(torch.autograd.Function):
    """nn.Dropout sites outside the blocks (HF/models/t5/modeling_t5.py:734,768)."""

    @staticmethod
    def forward(ctx, x, p, seed, seed_ptr):
        ctx.p, ctx.seed, ctx.seed_ptr = p, seed, seed_ptr
        return O.dropout_apply(x, p, seed, seed_ptr)

    @staticmethod
    @_backward_phase
    def backward(ctx, dy):
        return O.dropout_apply(dy, ctx.p, ctx.seed, ctx.seed_ptr), None, None, None


class ConcatEmbeddingsFn(torch.autograd.Function):
    """/root/reference/models/model.py:20-23: final LayerNorm of Swin (HF/models/swinv2/modeling_swinv2.py:969) and final
    RMSNorm of the frozen text encoder (HF/models/t5/modeling_t5.py:767) written straight into one [B, N_img + L_src, d] buffer
    (torch.cat costs no copy).  Gradient flows to the image branch only (the text encoder is frozen, model.py:14,20)."""

    @staticmethod
    def forward(ctx, img, ln_w, ln_b, ln_eps, lang, rms_w, rms_eps, B):
        n_img, d = img.shape[0] // B, img.shape[1]
        l_src = lang.shape[0] // B
        le = n_img + l_src
        buf = torch.empty(B, le, d, dtype=img.dtype, device=img.device)
        save = _needs_grad((img, ln_w, ln_b))
        _, mean, rstd = O.layernorm_fwd(img, ln_w, ln_b, ln_eps, out=buf, out_rows_per_group=n_img, out_group_stride=le * d,
                                        save_stats=save)
        O.rmsnorm_fwd(lang, rms_w, rms_eps, out=buf[:, n_img:], out_rows_per_group=l_src, out_group_stride=le * d, save_stats=False)
        if save:
            ctx.save_for_backward(img, ln_w, mean, rstd)
            ctx.geom = (n_img, le, d)
        return buf.view(B * le, d)

    @staticmethod
    @_backward_phase
    def backward(ctx, dbuf):
        img, ln_w, mean, rstd = ctx.saved_tensors
        n_img, le, d = ctx.geom
        dbuf = dbuf.contiguous()
        dimg, dg, db = O.layernorm_bwd(dbuf, img, ln_w, mean, rstd, dy_ld=d, dy_rows_per_group=n_img, dy_group_stride=le * d)
        return dimg, dg, db, None, None, None, None, None


# ------------------------------------------------------------------------------------------------
# decoder input embedding and LM head + loss
# ------------------------------------------------------------------------------------------------
class DecoderEmbedFn(torch.autograd.Function):
    """embed_tokens(_shift_right(labels)), HF/models/t5/modeling_t5.py:595-614,:682,:1089."""

    @staticmethod
    def forward(ctx, labels, table, cache, cd, start_id, pad_id):
        tab = cache.get([table], cd)
        y = O.embedding_fwd(labels, tab, shift_right=True, start_id=start_id, pad_id=pad_id)
        if _needs_grad((table,)):
            ctx.save_for_backward(labels)
            ctx.meta = (table.shape, start_id, pad_id)
        return y

    @staticmethod
    @_backward_phase
    def backward(ctx, dy):
        (labels,) = ctx.saved_tensors
        shape, start_id, pad_id = ctx.meta
        dtab = torch.zeros(shape, dtype=torch.float32, device=dy.device)
        O.embedding_bwd(labels, dy.contiguous(), dtab, shift_right=True, start_id=start_id, pad_id=pad_id)
        return None, dtab, None, None, None, None


LMHEAD_VOCAB_CHUNK = 8192      # backward recomputes the logits this many vocabulary columns at a time (scratch stays in L2)


class LMHeadLossFn(torch.autograd.Function):
    """final RMSNorm -> dropout (training) -> * alpha -> LM head -> CrossEntropyLoss(ignore_index=-100),
    HF/models/t5/modeling_t5.py:767-768,1105-1117.  alpha = d_model**-0.5, or 1 for T5 v1.1 (config.scale_decoder_outputs);
    `table` is lm_head.weight (shared.weight itself when tied).

    bf16 (hot path): the LM-head GEMM is fused with the cross entropy and vocab-tiled -- its epilogue reduces every 128 x 256
    logits tile to online-softmax partials straight out of TMEM, so the [rows, 32128] logits are never written; backward
    recomputes them one vocabulary chunk at a time into a chunk-sized scratch of d loss / d logits and feeds the two gradient
    GEMMs from it (dH accumulates in fp32, dE rows of the chunk are written once).
    fp32 (strict parity path): materialised logits + klab_ce_fwd / klab_ce_bwd."""

    @staticmethod
    def forward(ctx, x, ln_w, table, labels, cache, eps, p, seed, seed_ptr, alpha):
        cd = x.dtype
        V, d = table.shape
        tab = cache.get([table], cd)
        n, rstd = O.rmsnorm_fwd(x, ln_w, eps)
        if p > 0.0:
            n = O.dropout_apply(n, p, seed, seed_ptr)
        lab = labels.reshape(-1).contiguous()
        fused = cd == torch.bfloat16
        if fused:
            logits, vpad = None, 0
            lse, stats = O.lmhead_ce_fwd(n, tab, alpha, lab)
        else:
            vpad = (V + 7) // 8 * 8
            logits = O.linear_fwd(n, tab, alpha=alpha, ldd_pad=vpad)
            lse, stats = O.ce_fwd(logits, V, lab)
        if _needs_grad((x, ln_w, table)):
            ctx.save_for_backward(x, ln_w, table, lab, rstd, n, logits, lse, stats)
            ctx.cache, ctx.vpad, ctx.p, ctx.seed, ctx.seed_ptr, ctx.fused, ctx.alpha = cache, vpad, p, seed, seed_ptr, fused, alpha
            ctx.step_token = _StepToken()
        return stats[0].clone()

    @staticmethod
    @_backward_phase
    def backward(ctx, gloss):
        ctx.step_token.release()
        x, ln_w, table, lab, rstd, n, logits, lse, stats = ctx.saved_tensors
        V, d = table.shape
        tab = ctx.cache.get([table], x.dtype)
        g = gloss.reshape(1).to(torch.float32).contiguous()
        alpha = ctx.alpha
        if ctx.fused:
            rows = n.shape[0]
            chunk = min(LMHEAD_VOCAB_CHUNK, (V + 7) // 8 * 8)
            scratch = torch.empty(rows, chunk, dtype=torch.bfloat16, device=n.device)
            dn32 = torch.empty(rows, d, dtype=torch.float32, device=n.device)
            dtab = torch.empty(V, d, dtype=torch.float32, device=n.device)
            for v0 in range(0, V, chunk):
                vc = min(chunk, V - v0)
                dl = O.lmhead_ce_bwd_chunk(n, tab, alpha, lab, lse, stats, g, v0, vc, scratch)
                O.gemm(dl, tab[v0:v0 + vc], rows, d, vc, b_mn=True, out=dn32, alpha=alpha, accumulate=v0 > 0)      # dH (+)= dlogits E_chunk
                O.gemm(dl, n, vc, d, rows, a_mn=True, b_mn=True, out=dtab[v0:v0 + vc], alpha=alpha)                 # dE_chunk = dlogits^T H
            dn = O.cast(dn32, x.dtype)
        else:
            O.ce_bwd(logits, V, ctx.vpad, lab, lse, stats, g)            # logits now hold d loss / d logits
            dn = O.linear_dgrad(logits, tab, alpha=alpha)
            dtab = O.linear_wgrad(logits, n, alpha=alpha)
        if ctx.p > 0.0:
            dn = O.dropout_apply(dn, ctx.p, ctx.seed, ctx.seed_ptr)
        dx, dln = O.rmsnorm_bwd(dn, x, ln_w, rstd)
        return dx, dln, dtab, None, None, None, None, None, None, None


# ------------------------------------------------------------------------------------------------
# Swin-V2  (HF/models/swinv2/modeling_swinv2.py)
# ------------------------------------------------------------------------------------------------
class PatchEmbedFn(torch.autograd.Function):
    """Swinv2Embeddings: Conv2d(k = s = patch) as im2col + GEMM (+bias), then LayerNorm (:265-334)."""

    @staticmethod
    def forward(ctx, pixels, conv_w, conv_b, ln_w, ln_b, cache, cd, patch, eps):
        pm = O.patchify(pixels.contiguous().float(), patch, cd)
        w = cache.get([conv_w], cd)
        e = O.linear_fwd(pm, w, bias=conv_b)
        save = _needs_grad((conv_w, conv_b, ln_w, ln_b))
        y, mean, rstd = O.layernorm_fwd(e, ln_w, ln_b, eps, save_stats=save)
        if save:
            ctx.save_for_backward(pm, e, ln_w, mean, rstd)
            ctx.wshape = conv_w.shape
        return y

    @staticmethod
    @_backward_phase
    def backward(ctx, dy):
        pm, e, ln_w, mean, rstd = ctx.saved_tensors
        de, dg, db = O.layernorm_bwd(dy.contiguous(), e, ln_w, mean, rstd)
        dw = O.linear_wgrad(de, pm).view(ctx.wshape)
        dbias = O.colsum(de)
        return None, dw, dbias, dg, db, None, None, None, None


class PatchMergeFn(torch.autograd.Function):
    """Swinv2PatchMerging (:365-388): 2x2 gather -> Linear(4C, 2C, no bias) -> LayerNorm."""

    @staticmethod
    def forward(ctx, x, red_w, ln_w, ln_b, cache, B, res, eps):
        C_ = x.shape[1]
        g = O.patch_merge(x.contiguous(), B, res, C_)
        w = cache.get([red_w], x.dtype)
        r = O.linear_fwd(g, w)
        save = _needs_grad((x, red_w, ln_w, ln_b))
        y, mean, rstd = O.layernorm_fwd(r, ln_w, ln_b, eps, save_stats=save)
        if save:
            ctx.save_for_backward(g, r, red_w, ln_w, mean, rstd)
            ctx.meta = (cache, B, res, C_)
        return y

    @staticmethod
    @_backward_phase
    def backward(ctx, dy):
        g, r, red_w, ln_w, mean, rstd = ctx.saved_tensors
        cache, B, res, C_ = ctx.meta
        w = cache.get([red_w], g.dtype)
        dr, dg_, db_ = O.layernorm_bwd(dy.contiguous(), r, ln_w, mean, rstd)
        dgath = O.linear_dgrad(dr, w)
        dw = O.linear_wgrad(dr, g)
        dx = O.patch_merge(dgath, B, res, C_, scatter=True)
        return dx, dw, dg_, db_, None, None, None, None


def _swin_operands(c, params, cd, mode):
    (ls, w1, b1, w2, qw, qb, kw, vw, vb, pw, pb, g1, be1, f1w, f1b, f2w, f2b, g2, be2) = params
    f = getattr(c.cache, mode)
    return f([qw, kw, vw], cd), f([pw], cd), f([f1w], cd), f([f2w], cd)


def _swin_block_fwd_body(x, c, save, *params):
    """-> (out,) or (out, qkv, bias16, hidden, tab, ctx, lse, a, mean1, rstd1, h, m_pre, m_act, m2, mean2, rstd2)"""
    (ls, w1, b1, w2, qw, qb, kw, vw, vb, pw, pb, g1, be1, f1w, f1b, f2w, f2b, g2, be2) = params
    cd = x.dtype
    C_ = x.shape[1]
    wqkv, w_p, w_f1, w_f2 = _swin_operands(c, params, cd, "peek")
    bqkv = cat_vec([(qb, C_), (None, C_), (vb, C_)], x.device)            # key has no bias (:417)
    # the continuous position bias depends on weights only: side stream, joined before the attention kernel
    w1d, b1d, w2d = w1.detach(), b1.detach(), w2.detach()
    bias16, hidden, tab = _Side.run(lambda *_: O.swin_cpb_fwd(c.coords, c.index, w1d, b1d, w2d, c.heads, c.N), w1d, b1d, w2d)
    qkv = O.linear_fwd(x, wqkv, bias=bqkv)
    lsv = ls.detach().reshape(-1)
    q, k, v = qkv[:, :C_], qkv[:, C_:2 * C_], qkv[:, 2 * C_:]
    _Side.join()
    ctxt, lse = O.swin_attention_fwd(q, k, v, c.B, c.res, c.heads, c.hd, c.w, c.shift, lsv, bias16)
    a = O.linear_fwd(ctxt, w_p, bias=pb)
    h, mean1, rstd1 = O.layernorm_fwd(a, g1, be1, c.eps, residual=x, save_stats=save)       # res-post-norm (:707-708)
    m_pre = torch.empty(x.shape[0], 4 * C_, dtype=cd, device=x.device) if save else None
    m_act = O.linear_fwd(h, w_f1, bias=f1b, act=L.ACT_GELU_SAVE_GRAD if save else L.ACT_GELU, aux_out=m_pre)   # m_pre := gelu'(fc1 output)
    m2 = O.linear_fwd(m_act, w_f2, bias=f2b)
    out, mean2, rstd2 = O.layernorm_fwd(m2, g2, be2, c.eps, residual=h, save_stats=save)      # :712
    if not save:
        return (out,)
    return (out, qkv, bias16, hidden, tab, ctxt, lse, a, mean1, rstd1, h, m_pre, m_act, m2, mean2, rstd2)


_N_SWIN_ACTS = 15
_N_SWIN_GRADS = 19            # one per parameter of a block, in flat_params() order


def _swin_block_bwd_body(dout, x, *rest):
    """rest = saved activations (15), [accumulators (22): the static outputs of an earlier run of this region,] c, params (19)
    -> (dx, 19 parameter gradients, dwqkv, dbqkv, flat).  Every parameter gradient is a slice of `flat` (see _flat_grads); dwqkv /
    dbqkv are the slices the q / k / v weight and bias gradients are views of.  With accumulators every parameter gradient is ADDED
    into the given buffer by the kernel that produces it (GEMM epilogue / norm / colsum / CPB kernels all have an accumulate mode)
    and the same buffers are returned."""
    (qkv, bias16, hidden, tab, ctxt, lse, a, mean1, rstd1, h, m_pre, m_act, m2, mean2, rstd2), rest = rest[:_N_SWIN_ACTS], rest[_N_SWIN_ACTS:]
    acc = len(rest) > 1 + _N_SWIN_GRADS
    if acc:
        go, rest = rest[:_N_SWIN_GRADS + 3], rest[_N_SWIN_GRADS + 3:]
        (o_ls, o_w1, o_b1, o_w2, _gq, _gbq, _gk, _gv, _gbv, o_pw, o_pb, o_g1, o_be1, o_f1w, o_f1b, o_f2w, o_f2b, o_g2, o_be2, o_wqkv, o_bqkv,
         flat) = go
    c, params = rest[0], rest[1:]
    (ls, w1, b1, w2, qw, qb, kw, vw, vb, pw, pb, g1, be1, f1w, f1b, f2w, f2b, g2, be2) = params
    cd = x.dtype
    C_ = x.shape[1]
    wqkv, w_p, w_f1, w_f2 = _swin_operands(c, params, cd, "peek")
    if not acc:
        flat, (o_ls, o_w1, o_b1, o_w2, o_wqkv, o_bqkv, o_pw, o_pb, o_g1, o_be1, o_f1w, o_f1b, o_f2w, o_f2b, o_g2, o_be2) = _flat_grads(
            [(c.heads,), tuple(w1.shape), tuple(b1.shape), tuple(w2.shape), (3 * C_, C_), (3 * C_,), (C_, C_), (C_,), (C_,), (C_,),
             (4 * C_, C_), (4 * C_,), (C_, 4 * C_), (C_,), (C_,), (C_,)], x.device)

    def wg(t):                                                           # keyword arguments of a weight-gradient GEMM into `t`
        return dict(out=t, accumulate=acc)

    dm2, dg2, dbe2 = O.layernorm_bwd(dout, m2, g2, mean2, rstd2, dgamma=o_g2, dbeta=o_be2, accumulate=acc)
    dm_pre = O.linear_dgrad(dm2, w_f2, act=L.ACT_MUL_AUX, aux_in=m_pre)                  # m_pre holds gelu'(fc1 output), saved by the forward epilogue
    df2w = _wgrad(dm2, m_act, **wg(o_f2w))
    df2b = _Side.run(O.colsum, dm2, out=o_f2b, accumulate=acc)
    dh = O.linear_dgrad(dm_pre, w_f1, residual=dout)                     # + residual path of the second norm
    df1w = _wgrad(dm_pre, h, **wg(o_f1w))
    df1b = _Side.run(O.colsum, dm_pre, out=o_f1b, accumulate=acc)
    da, dg1, dbe1 = O.layernorm_bwd(dh, a, g1, mean1, rstd1, dgamma=o_g1, dbeta=o_be1, accumulate=acc)
    dctx = O.linear_dgrad(da, w_p)
    dpw = _wgrad(da, ctxt, **wg(o_pw))
    dpb = _Side.run(O.colsum, da, out=o_pb, accumulate=acc)
    dqkv = torch.empty_like(qkv)
    q, k, v = qkv[:, :C_], qkv[:, C_:2 * C_], qkv[:, 2 * C_:]
    lsv = ls.detach().reshape(-1)
    dbias, dls = O.swin_attention_bwd(q, k, v, ctxt, dctx, dqkv[:, :C_], dqkv[:, C_:2 * C_], dqkv[:, 2 * C_:], c.B, c.res,
                                      c.heads, c.hd, c.w, c.shift, lsv, bias16, lse, dls_out=None if acc else o_ls.view(-1))
    if acc:
        O.colsum(dls.view(1, -1), out=o_ls.view(-1))                     # o_ls += dls (a one-row column sum)
    dls = o_ls.view(-1)
    w2d = w2.detach()                                                    # position-bias MLP gradients: off the critical path
    trio = (o_w1, o_b1, o_w2)
    dw1, db1, dw2 = _Side.run(lambda *_: O.swin_cpb_bwd(c.coords, c.index, w2d, hidden, tab, dbias, c.heads, c.N,
                                                         acc_into=trio if acc else None, out=None if acc else trio), dbias, hidden, tab, w2d)
    dx = O.linear_dgrad(dqkv, wqkv, residual=dh)                          # + residual path of the first norm
    dwqkv = _wgrad(dqkv, x, **wg(o_wqkv))
    dbqkv = _Side.run(O.colsum, dqkv, out=o_bqkv, accumulate=acc)
    _Side.join()
    return (dx, dls.view(ls.shape), dw1, db1, dw2, dwqkv[:C_], dbqkv[:C_], dwqkv[C_:2 * C_], dwqkv[2 * C_:], dbqkv[2 * C_:],
            dpw, dpb, dg1, dbe1, df1w, df1b, df2w, df2b, dg2, dbe2, dwqkv, dbqkv, flat)


class SwinBlockFn(torch.autograd.Function):
    """One Swinv2Layer (:662-715) with Swinv2SelfAttention (:421-487) inlined.
    params: logit_scale, cpb_w1, cpb_b1, cpb_w2, q_w, q_b, k_w, v_w, v_b, proj_w, proj_b, ln1_w, ln1_b, fc1_w, fc1_b, fc2_w, fc2_b,
            ln2_w, ln2_b"""

    @staticmethod
    def forward(ctx, c, x, *params):
        save = _needs_grad((x,) + tuple(params))
        _swin_operands(c, params, x.dtype, "get")
        x = x.contiguous()
        outs, graphed = POOL.run(("swf", id(c), save), _swin_block_fwd_body, (x,), (c, save) + tuple(params),
                                 allow_graph=not c.busy)
        if save:
            ctx.c = c
            ctx.graphed = graphed
            ctx.save_for_backward(x, *params)
            ctx.acts = outs[1:]
            if graphed:
                c.busy = True
                ctx.token = _Token(c)
        return outs[0]

    @staticmethod
    @_backward_phase
    def backward(ctx, dout):
        c = ctx.c
        x, *params = ctx.saved_tensors
        acts, ctx.acts = ctx.acts, None
        # The reference's optimizer does not own the image model (train.py:28), so with --image_model_train its gradients are
        # never zeroed and accumulate step after step (SURVEY.md 9 Q3): autograd would run one `grad += new` kernel per
        # parameter per step (456 tiny launches).  When every parameter's .grad still IS the static gradient buffer this region
        # handed out last time, the accumulating variant of the region adds the new gradients into those buffers inside the
        # kernels that produce them, .grad is reset, and autograd re-adopts the very same buffers: no copies, no add kernels,
        # hooks (the data-parallel reducer) fire as usual.
        prev = getattr(c, "bwd_static", None)
        use_acc = (ctx.graphed and prev is not None and ACCUMULATE_IN_PLACE and
                   all(p.grad is not None and p.grad.data_ptr() == o.data_ptr() and p.grad.shape == o.shape
                       for p, o in zip(params, prev[1:1 + _N_SWIN_GRADS])))
        if use_acc:
            for p in params:
                p.grad = None
            outs, graphed = POOL.run(("swba", id(c)), _swin_block_bwd_body, (dout.contiguous(), x) + tuple(acts) + tuple(prev[1:]),
                                     (c,) + tuple(params), allow_graph=True)
        else:
            if ctx.graphed:
                _detach_aliased_grads(params)
            outs, graphed = POOL.run(("swb", id(c)), _swin_block_bwd_body, (dout.contiguous(), x) + tuple(acts), (c,) + tuple(params),
                                     allow_graph=ctx.graphed)
            c.bwd_static = outs if graphed else None
            if graphed and ACCUMULATE_IN_PLACE:
                # first captured run with gradients already accumulated elsewhere: fold the old values into the static buffers
                # once (the add autograd was about to do anyway) so that, from the next step on, .grad IS the static buffer
                olds = [p.grad for p in params]
                news = list(outs[1:1 + _N_SWIN_GRADS])
                if all(g is not None and g.shape == o.shape and g.dtype == o.dtype and g.device == o.device for g, o in zip(olds, news)):
                    torch._foreach_add_(news, olds)
                    for p in params:
                        p.grad = None
        tok, ctx.token = getattr(ctx, "token", None), None
        if tok is not None:
            tok.release()
        _publish_flat(params, outs[-1], all(p.grad is None for p in params))
        return (None,) + _grad_outputs(outs[:1 + _N_SWIN_GRADS], graphed or use_acc)
