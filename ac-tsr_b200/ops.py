"""torch.autograd.Function wrappers over the C ABI (include/acsr.h).

PyTorch is plumbing here: it owns device memory, the stream and the autograd tape; every op
below launches hand-written sm_100a kernels from libacsr.so.  Tensors must be CUDA, contiguous,
float32 (ids int64) -- anything else raises; there is no CPU or eager fallback.
"""
import ctypes

import numpy as np
import torch

from ._lib import LIB, AcsrError

ACT_IDS = {'gelu': 0, 'relu': 1, 'swish': 2, 'tanh': 3, 'sigmoid': 4}
COMBINE_IDS = {'gate': 0, 'fixed': 1, 'annealing': 2}
RICH_IDS = {'none': 0, 'fixed': 1, 'trainable': 2}


def _p(t, dtype=torch.float32):
    """device pointer of a tensor (None -> NULL) after checking the ABI's layout contract."""
    if t is None:
        return None
    if not t.is_cuda:
        raise AcsrError('AC-SASRec hot path needs CUDA tensors (got %s); there is no CPU fallback' % t.device)
    if t.dtype != dtype:
        raise AcsrError('expected dtype %s, got %s' % (dtype, t.dtype))
    if not t.is_contiguous():
        raise AcsrError('tensor must be contiguous')
    return t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _c(t):
    return None if t is None else t.contiguous()


def _wants_grad(t):
    """False only for a LEAF tensor whose requires_grad is off right now.  The reference trainer routes its two backward passes by
    toggling requires_grad on the parameters between them (trainer.py:672-686): the graph was built with every parameter
    trainable, so ctx.needs_input_grad still says True, but autograd drops a gradient that arrives at a leaf with
    requires_grad False -- computing it would be wasted work (half of all weight-gradient launches of a step)."""
    return t is not None and (t.requires_grad or not t.is_leaf)


_DIRECT_GRAD = [False]


class direct_param_grads:
    """Inside this context the backward kernels accumulate parameter gradients STRAIGHT into `param.grad` when the parameter is a
    leaf that owns a gradient buffer (the trainer's flat gradient) and return None for it: the kernels add with atomics anyway,
    so the zero-filled temporary and autograd's `grad += temporary` -- two more launches per parameter and pass -- disappear.
    The trainer's step uses it; everywhere else (tests, torch.autograd.grad) gradients are returned the usual way."""

    def __enter__(self):
        self.prev = _DIRECT_GRAD[0]
        _DIRECT_GRAD[0] = True

    def __exit__(self, *a):
        _DIRECT_GRAD[0] = self.prev


def _grad_sink(t):
    """the buffer a backward kernel may accumulate t's gradient into directly, or None"""
    if _DIRECT_GRAD[0] and t is not None and t.is_leaf and t.requires_grad and t.grad is not None and t.grad.is_contiguous():
        return t.grad
    return None


def _param_grad_buffers(params):
    """gradient destinations of a backward kernel for the given parameter tensors (None entries allowed) ->
    (buffers handed to the kernel, gradients returned to autograd).  A parameter whose gradient autograd would drop gets no
    buffer (the kernels skip NULL destinations); one with a sink accumulates in place; the rest share ONE zero-filled block."""
    bufs, rets, need = [None] * len(params), [None] * len(params), []
    for i, t in enumerate(params):
        if t is None or not _wants_grad(t):
            continue
        sink = _grad_sink(t)
        if sink is not None:
            bufs[i] = sink
        else:
            need.append(i)
    if need:
        sizes = [(params[i].numel() + 3) // 4 * 4 for i in need]
        block = torch.zeros(sum(sizes), dtype=torch.float32, device=params[need[0]].device)
        off = 0
        for i, n in zip(need, sizes):
            bufs[i] = rets[i] = block[off:off + params[i].numel()].view(params[i].shape)
            off += n
    return bufs, rets


class DeviceRng:
    """{seed, step} in device memory; kernels read it so CUDA-graph replays draw fresh masks."""

    def __init__(self, seed, device):
        self.state = torch.tensor([int(seed) & 0x7fffffffffffffff, 0], dtype=torch.int64, device=device)

    @property
    def ptr(self):
        return self.state.data_ptr()

    def advance(self):
        LIB.call('acsr_rng_advance', self.ptr, _stream())


# ------------------------------------------------------------------------------------------
class EmbedLnDropoutFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, item_seq, table, pos_emb, ln_w, ln_b, eps, p, mask, rng, rng_stream):
        B, L = item_seq.shape
        V, d = table.shape
        item_seq = item_seq.contiguous()
        out = torch.empty((B, L, d), dtype=torch.float32, device=table.device)
        stats = torch.empty((B * L, 2), dtype=torch.float32, device=table.device)
        mask = _c(mask)
        LIB.call('acsr_embed_ln_dropout_fwd', _p(item_seq, torch.int64), _p(table), _p(pos_emb), _p(ln_w), _p(ln_b),
                 eps, B * L, L, d, V, p, _p(mask), rng.ptr if rng is not None else None, rng_stream,
                 _p(out), _p(stats), _stream())
        ctx.save_for_backward(item_seq, table, pos_emb, ln_w, stats, mask)
        ctx.meta = (B, L, d, V, p, rng, rng_stream)
        return out

    @staticmethod
    def backward(ctx, d_out):
        item_seq, table, pos_emb, ln_w, stats, mask = ctx.saved_tensors
        B, L, d, V, p, rng, rng_stream = ctx.meta
        if not (_wants_grad(table) or _wants_grad(pos_emb) or _wants_grad(ln_w)):      # the attacked-loss pass of the routed backward
            return None, None, None, None, None, None, None, None, None, None
        d_out = d_out.contiguous()
        d_table = torch.zeros_like(table)
        d_pos = torch.zeros_like(pos_emb) if pos_emb is not None else None
        d_w = torch.zeros_like(ln_w)
        d_b = torch.zeros_like(ln_w)
        LIB.call('acsr_embed_ln_dropout_bwd', _p(d_out), _p(item_seq, torch.int64), _p(table), _p(pos_emb), _p(ln_w),
                 _p(stats), B * L, L, d, V, p, _p(mask), rng.ptr if rng is not None else None, rng_stream,
                 _p(d_table), _p(d_pos), _p(d_w), _p(d_b), _stream())
        return None, d_table, d_pos, d_w, d_b, None, None, None, None, None


class BiasDropoutResLnFn(torch.autograd.Function):
    """LN(dropout(h + bias) + res)  -- layers.py:681-683 / 794-796."""

    @staticmethod
    def forward(ctx, h, bias, res, ln_w, ln_b, eps, p, mask, rng, rng_stream):
        h, res, mask = h.contiguous(), res.contiguous(), _c(mask)
        d = h.shape[-1]
        T = h.numel() // d
        out = torch.empty_like(h)
        stats = torch.empty((T, 2), dtype=torch.float32, device=h.device)
        LIB.call('acsr_bias_dropout_res_ln_fwd', _p(h), _p(bias), _p(res), _p(ln_w), _p(ln_b), eps, T, d, T, p, _p(mask),
                 rng.ptr if rng is not None else None, rng_stream, _p(out), _p(stats), _stream())
        ctx.save_for_backward(h, bias, res, ln_w, stats, mask)
        ctx.meta = (T, d, p, rng, rng_stream)
        ctx.ln_b_ref = ln_b
        return out

    @staticmethod
    def backward(ctx, d_out):
        h, bias, res, ln_w, stats, mask = ctx.saved_tensors
        T, d, p, rng, rng_stream = ctx.meta
        d_out = d_out.contiguous()
        d_h = torch.empty_like(h)
        d_res = torch.empty_like(h)
        (b_bias, b_w, b_b), (d_bias, d_w, d_b) = _param_grad_buffers([bias, ln_w, ctx.ln_b_ref])
        LIB.call('acsr_bias_dropout_res_ln_bwd', _p(d_out), _p(h), _p(bias), _p(res), _p(ln_w), _p(stats), T, d, T, T, T, p,
                 _p(mask), rng.ptr if rng is not None else None, rng_stream, _p(d_h), _p(d_res), _p(b_bias), _p(b_w),
                 _p(b_b), _stream())
        return d_h, d_bias, d_res, d_w, d_b, None, None, None, None, None


class BiasActFn(torch.autograd.Function):
    """act(h + bias)  -- layers.py:776-792."""

    @staticmethod
    def forward(ctx, h, bias, act):
        h = h.contiguous()
        n = h.shape[-1]
        T = h.numel() // n
        out = torch.empty_like(h)
        LIB.call('acsr_bias_act_fwd', _p(h), _p(bias), T, n, act, _p(out), _stream())
        ctx.save_for_backward(h, bias)
        ctx.meta = (T, n, act)
        return out

    @staticmethod
    def backward(ctx, d_out):
        h, bias = ctx.saved_tensors
        T, n, act = ctx.meta
        d_out = d_out.contiguous()
        d_h = torch.empty_like(h)
        (b_bias,), (d_bias,) = _param_grad_buffers([bias])
        LIB.call('acsr_bias_act_bwd', _p(d_out), _p(h), _p(bias), T, n, act, T, T, _p(d_h), _p(b_bias), _stream())
        return d_h, d_bias, None


class GatherLastFn(torch.autograd.Function):
    """rows [0,B) = x_att[b, len-1], rows [B,2B) = x_cal[b, len-1]  (abstract_recommender.py:130-134)."""

    @staticmethod
    def forward(ctx, x_att, x_cal, item_len):
        B, L, d = x_cal.shape
        x_cal = x_cal.contiguous()
        x_att = _c(x_att)
        item_len = item_len.contiguous()
        rows = 2 * B if x_att is not None else B
        out = torch.empty((rows, d), dtype=torch.float32, device=x_cal.device)
        LIB.call('acsr_gather_last_fwd', _p(x_att), _p(x_cal), _p(item_len, torch.int64), B, L, d, _p(out), _stream())
        ctx.save_for_backward(item_len)
        ctx.meta = (B, L, d, x_att is not None)
        return out

    @staticmethod
    def backward(ctx, d_out):
        (item_len,) = ctx.saved_tensors
        B, L, d, has_att = ctx.meta
        d_out = d_out.contiguous()
        d_cal = torch.zeros((B, L, d), dtype=torch.float32, device=d_out.device)
        d_att = torch.zeros_like(d_cal) if has_att else None
        LIB.call('acsr_gather_last_bwd', _p(d_out), _p(item_len, torch.int64), B, L, d, _p(d_att), _p(d_cal), _stream())
        return d_att, d_cal, None


def attn_workspace(B, L, H, n_streams, device):
    """scratch for the attention backward of sequences longer than 64 (attn_long.cu): as many sequences' worth as fit
    under ACSR_WORKSPACE_MB (default 4096); the library walks the batch in chunks of that many sequences."""
    if L <= 64:
        return
    import os
    per_seq = LIB.query('acsr_attn_workspace_bytes', int(L), int(H), int(n_streams))
    cap = int(os.environ.get('ACSR_WORKSPACE_MB', 4096)) << 20
    LIB.ensure_workspace(max(per_seq, min(B * per_seq, cap)), device)


class AttnOpts:
    """static options of one fused-attention call (mirrors the AttackR* constructor flags)."""

    def __init__(self, n_heads, two_level, combine_option, rich_mode, p_attn, bidirectional=False, plain=False):
        self.n_heads = n_heads
        # the ABI's `two_level` argument carries three flags: bit 0 two_level, bit 1 bidirectional attention mask (AcBERT4Rec),
        # bit 2 the transformer_layers.py variant without the re-normalising softmaxes (ACSSEPT), see ACSR_ATTN_PLAIN
        self.two_level = int(bool(two_level)) | (2 if bidirectional else 0) | (4 if plain else 0)
        self.combine = COMBINE_IDS[combine_option]
        self.rich = RICH_IDS.get(rich_mode, 0)
        self.p_attn = float(p_attn)


class AttnCalibFn(torch.autograd.Function):
    """fused spatial + adversarial calibrated attention; returns (ctx_att|None, ctx_cal, pen_sq)."""

    @staticmethod
    def forward(ctx, mq, mk, mv, aq, ak, gate_logit, key_ids, order_w, order_b, dist_w, dist_b, scalar, rich_ratio,
                opts, comb_scalar, p_attn, rand, rng, rng_stream, need_att, want_probs):
        B, L, d = mq.shape
        H = opts.n_heads
        dh = d // H
        ctx.set_materialize_grads(False)     # unused outputs arrive as None -> the kernel skips that branch
        mq, mk, mv, aq, ak = (t.contiguous() for t in (mq, mk, mv, aq, ak))
        gate_logit = _c(gate_logit)
        key_ids = key_ids.contiguous()
        D1, D2, D3, noise = (_c(rand.get(k)) if rand else None for k in ('D1', 'D2', 'D3', 'noise'))
        dev = mq.device
        ctx_cal = torch.empty((B, L, d), dtype=torch.float32, device=dev)
        ctx_att = torch.empty_like(ctx_cal) if need_att else None
        pen = torch.zeros(1, dtype=torch.float64, device=dev)
        probs = torch.empty((6, B, H, L, L), dtype=torch.float32, device=dev) if want_probs else None
        rngp = rng.ptr if rng is not None else None
        LIB.call('acsr_attn_calib_fwd', _p(mq), _p(mk), _p(mv), _p(aq), _p(ak), _p(gate_logit), _p(key_ids, torch.int64),
                 _p(order_w), _p(order_b), _p(dist_w), _p(dist_b), _p(scalar), B, L, H, dh,
                 opts.two_level, opts.combine, float(comb_scalar), opts.rich, _p(rich_ratio),
                 p_attn, _p(D1), _p(D2), _p(D3), _p(noise), rngp, rng_stream,
                 _p(ctx_att), _p(ctx_cal), pen.data_ptr(), _p(probs), None, None, _stream())
        ctx.save_for_backward(mq, mk, mv, aq, ak, gate_logit, key_ids, order_w, order_b, dist_w, dist_b, scalar, rich_ratio,
                              D1, D2, D3, noise)
        ctx.meta = (B, L, H, dh, opts, float(comb_scalar), p_attn, rng, rng_stream, need_att)
        pen32 = pen.to(torch.float32)
        ctx.mark_non_differentiable(*([probs] if probs is not None else []))
        return ctx_att, ctx_cal, pen32, probs

    @staticmethod
    def backward(ctx, d_att, d_cal, d_pen, _d_probs):
        (mq, mk, mv, aq, ak, gate_logit, key_ids, order_w, order_b, dist_w, dist_b, scalar, rich_ratio,
         D1, D2, D3, noise) = ctx.saved_tensors
        B, L, H, dh, opts, comb_scalar, p_attn, rng, rng_stream, need_att = ctx.meta
        d_att = _c(d_att) if need_att else None
        d_cal = _c(d_cal)
        d_pen = _c(d_pen)
        z = torch.zeros_like
        d_mq, d_mk, d_mv, d_aq, d_ak = (torch.empty_like(mq) for _ in range(5))
        d_gate = z(gate_logit) if gate_logit is not None else None
        # the calibrator parameters: straight into their .grad when the trainer asks for it, dropped (NULL) when the routed backward
        # would discard them, else one shared zero-filled block
        (b_ow, b_ob, b_dw, b_db, b_sc, b_rr), (d_ow, d_ob, d_dw, d_db, d_sc, d_rr) = _param_grad_buffers(
            [order_w, order_b, dist_w, dist_b, scalar, rich_ratio])
        attn_workspace(B, L, H, 1, mq.device)
        LIB.call('acsr_attn_calib_bwd', _p(d_att), _p(d_cal), _p(d_pen), _p(mq), _p(mk), _p(mv), _p(aq), _p(ak),
                 _p(gate_logit), _p(key_ids, torch.int64), _p(order_w), _p(order_b), _p(dist_w), _p(dist_b), _p(scalar),
                 B, L, H, dh, opts.two_level, opts.combine, comb_scalar, opts.rich, _p(rich_ratio),
                 p_attn, _p(D1), _p(D2), _p(D3), _p(noise), rng.ptr if rng is not None else None, rng_stream,
                 _p(d_mq), _p(d_mk), _p(d_mv), _p(d_aq), _p(d_ak), _p(d_gate), _p(b_ow), _p(b_ob), _p(b_dw), _p(b_db),
                 _p(b_sc), _p(b_rr), None, None, _stream())
        return (d_mq, d_mk, d_mv, d_aq, d_ak, d_gate, None, d_ow, d_ob, d_dw, d_db, d_sc, d_rr,
                None, None, None, None, None, None, None, None)


# ------------------------------------------------------------------------------------------
# ACTiSASRec: time-interval aware keys / values (timeaware.cu) around the fused attention
# ------------------------------------------------------------------------------------------
def time_matrix(time_seq, time_span):
    """actisasrec.py:146-155: [B, L] time stamps -> int32 [B, L, L] clipped intervals"""
    ts = time_seq.to(torch.float32).contiguous()
    B, L = ts.shape
    out = torch.empty((B, L, L), dtype=torch.int32, device=ts.device)
    LIB.call('acsr_time_matrix', _p(ts), B, L, int(time_span), _p(out, torch.int32), _stream())
    return out


class PairSpec:
    """everything of the pair embedding E[b,i,j,c] = P[j,c]*Dp[b,j,c] + T[t[b,i,j],c]*Dt[b,i,j,c] except the two tables"""

    def __init__(self, tmat, n_heads, p, Dp=None, Dt=None, rng=None, stream_p=0, stream_t=0):
        self.tmat, self.H, self.p = tmat.contiguous(), int(n_heads), float(p)
        self.Dp, self.Dt = _c(Dp), _c(Dt)
        self.rng, self.stream_p, self.stream_t = rng, int(stream_p), int(stream_t)

    def args(self, B, L, d, span1):
        return (_p(self.tmat, torch.int32), B, L, self.H, d // self.H, span1, self.p, _p(self.Dp), _p(self.Dt),
                self.rng.ptr if (self.rng is not None and self.p > 0) else None, self.stream_p, self.stream_t)


def _pair_score(x, P, T, spec, causal):
    B, L, d = x.shape
    out = torch.empty((B, spec.H, L, L), dtype=torch.float32, device=x.device)
    a = spec.args(B, L, d, T.shape[0])
    LIB.call('acsr_pair_score', _p(x), _p(P), _p(T), *a, int(causal), _p(out), _stream())
    return out


def _pair_context(prob, P, T, spec, d):
    B, H, L, _ = prob.shape
    y = torch.empty((B, L, d), dtype=torch.float32, device=prob.device)
    a = spec.args(B, L, d, T.shape[0])
    LIB.call('acsr_pair_context', _p(prob), _p(P), _p(T), *a, 0, _p(y), _stream())
    return y


def _pair_wgrad(a_mat, v, P, T, spec):
    B, L, d = v.shape
    dP, dT = torch.zeros_like(P), torch.zeros_like(T)
    a = spec.args(B, L, d, T.shape[0])
    LIB.call('acsr_pair_wgrad', _p(a_mat), _p(v), a[0], *a[1:], _p(dP), _p(dT), _stream())
    return dP, dT


class PairScoreFn(torch.autograd.Function):
    """s[b,h,i,j] = q_i . (posK_j + timeK[t_ij]) per head, with the reference's element-wise dropout of both embeddings
    (actisasrec.py:120-123, transformer_layers.py:1128-1134); the [B,L,L,d] gather never exists."""

    @staticmethod
    def forward(ctx, x, P, T, spec, causal):
        x, P, T = x.contiguous(), P.contiguous(), T.contiguous()
        ctx.save_for_backward(x, P, T)
        ctx.spec, ctx.causal = spec, bool(causal)
        return _pair_score(x, P, T, spec, causal)

    @staticmethod
    def backward(ctx, ds):
        x, P, T = ctx.saved_tensors
        ds = (torch.tril(ds) if ctx.causal else ds).contiguous()       # pairs j > i were not computed: they carry no gradient
        dx = _pair_context(ds, P, T, ctx.spec, x.shape[-1]) if ctx.needs_input_grad[0] else None
        dP = dT = None
        if (ctx.needs_input_grad[1] and _wants_grad(P)) or (ctx.needs_input_grad[2] and _wants_grad(T)):
            dP, dT = _pair_wgrad(ds, x, P, T, ctx.spec)
        return dx, dP, dT, None, None


class PairContextFn(torch.autograd.Function):
    """y[b,i,:] = sum_j prob[b,h,i,j] (posV_j + timeV[t_ij]) (transformer_layers.py:1088-1091)"""

    @staticmethod
    def forward(ctx, prob, P, T, spec):
        prob, P, T = prob.contiguous(), P.contiguous(), T.contiguous()
        ctx.save_for_backward(prob, P, T)
        ctx.spec = spec
        return _pair_context(prob, P, T, spec, P.shape[1])

    @staticmethod
    def backward(ctx, dy):
        prob, P, T = ctx.saved_tensors
        dy = dy.contiguous()
        dprob = _pair_score(dy, P, T, ctx.spec, 0) if ctx.needs_input_grad[0] else None
        dP = dT = None
        if (ctx.needs_input_grad[1] and _wants_grad(P)) or (ctx.needs_input_grad[2] and _wants_grad(T)):
            dP, dT = _pair_wgrad(prob, dy, P, T, ctx.spec)
        return dprob, dP, dT, None


class AttnCalibTiFn(torch.autograd.Function):
    """AttnCalibFn with an additive raw-score bias and the attacked / final calibrated attention matrices as differentiable
    outputs -> (ctx_att|None, ctx_cal, pen_sq, prob_att|None, prob_cal).  transformer_layers.py variant, L <= 64."""

    @staticmethod
    def forward(ctx, s_bias, mq, mk, mv, aq, ak, gate_logit, key_ids, order_w, order_b, dist_w, dist_b, scalar, rich_ratio,
                opts, comb_scalar, p_attn, rand, rng, rng_stream, need_att):
        B, L, d = mq.shape
        H = opts.n_heads
        dh = d // H
        ctx.set_materialize_grads(False)
        s_bias, mq, mk, mv, aq, ak = (t.contiguous() for t in (s_bias, mq, mk, mv, aq, ak))
        gate_logit = _c(gate_logit)
        key_ids = key_ids.contiguous()
        D1, D2, D3, noise = (_c(rand.get(k)) if rand else None for k in ('D1', 'D2', 'D3', 'noise'))
        dev = mq.device
        ctx_cal = torch.empty((B, L, d), dtype=torch.float32, device=dev)
        ctx_att = torch.empty_like(ctx_cal) if need_att else None
        # without the attacked stream (gate / annealing) the kernel only visits the keys in play: the rest of prob_cal is zero
        prob_cal = (torch.empty if need_att else torch.zeros)((B, H, L, L), dtype=torch.float32, device=dev)
        prob_att = torch.empty_like(prob_cal) if need_att else None
        pen = torch.zeros(1, dtype=torch.float64, device=dev)
        LIB.call('acsr_attn_calib_ti_fwd', _p(s_bias), _p(mq), _p(mk), _p(mv), _p(aq), _p(ak), _p(gate_logit),
                 _p(key_ids, torch.int64), _p(order_w), _p(order_b), _p(dist_w), _p(dist_b), _p(scalar), B, L, H, dh,
                 opts.two_level, opts.combine, float(comb_scalar), opts.rich, _p(rich_ratio),
                 p_attn, _p(D1), _p(D2), _p(D3), _p(noise), rng.ptr if rng is not None else None, rng_stream,
                 _p(ctx_att), _p(ctx_cal), pen.data_ptr(), _p(prob_att), _p(prob_cal), _stream())
        ctx.save_for_backward(s_bias, mq, mk, mv, aq, ak, gate_logit, key_ids, order_w, order_b, dist_w, dist_b, scalar,
                              rich_ratio, D1, D2, D3, noise)
        ctx.meta = (B, L, H, dh, opts, float(comb_scalar), p_attn, rng, rng_stream, need_att)
        return ctx_att, ctx_cal, pen.to(torch.float32), prob_att, prob_cal

    @staticmethod
    def backward(ctx, d_att, d_cal, d_pen, d_pa, d_pc):
        (s_bias, mq, mk, mv, aq, ak, gate_logit, key_ids, order_w, order_b, dist_w, dist_b, scalar, rich_ratio,
         D1, D2, D3, noise) = ctx.saved_tensors
        B, L, H, dh, opts, comb_scalar, p_attn, rng, rng_stream, need_att = ctx.meta
        d_att = _c(d_att) if need_att else None
        d_pa = _c(d_pa) if need_att else None
        d_cal, d_pen, d_pc = _c(d_cal), _c(d_pen), _c(d_pc)
        z = torch.zeros_like
        d_mq, d_mk, d_mv, d_aq, d_ak = (torch.empty_like(mq) for _ in range(5))
        d_gate = z(gate_logit) if gate_logit is not None else None
        (b_ow, b_ob, b_dw, b_db, b_sc, b_rr), (d_ow, d_ob, d_dw, d_db, d_sc, d_rr) = _param_grad_buffers(
            [order_w, order_b, dist_w, dist_b, scalar, rich_ratio])
        d_sb = z(s_bias)
        LIB.call('acsr_attn_calib_ti_bwd', _p(d_att), _p(d_cal), _p(d_pen), _p(d_pa), _p(d_pc), _p(s_bias), _p(mq), _p(mk),
                 _p(mv), _p(aq), _p(ak), _p(gate_logit), _p(key_ids, torch.int64), _p(order_w), _p(order_b), _p(dist_w),
                 _p(dist_b), _p(scalar), B, L, H, dh, opts.two_level, opts.combine, comb_scalar, opts.rich, _p(rich_ratio),
                 p_attn, _p(D1), _p(D2), _p(D3), _p(noise), rng.ptr if rng is not None else None, rng_stream,
                 _p(d_mq), _p(d_mk), _p(d_mv), _p(d_aq), _p(d_ak), _p(d_gate), _p(b_ow), _p(b_ob), _p(b_dw), _p(b_db),
                 _p(b_sc), _p(b_rr), _p(d_sb), _stream())
        return (d_sb, d_mq, d_mk, d_mv, d_aq, d_ak, d_gate, None, d_ow, d_ob, d_dw, d_db, d_sc, d_rr,
                None, None, None, None, None, None, None)


# ------------------------------------------------------------------------------------------
# full-catalogue logits on tcgen05
# ------------------------------------------------------------------------------------------
def logits_num_chunks(M, V, d=64):
    return LIB.query('acsr_logits_num_chunks_d', int(M), int(V), int(d))


def ce_partial(out, table, passes=3):
    """-> partial [M, n_chunks, 2] (max, sumexp) over this table (shard)."""
    M, d = out.shape
    V = table.shape[0]
    part = torch.empty((M, logits_num_chunks(M, V, d), 2), dtype=torch.float32, device=out.device)
    LIB.call('acsr_logits_ce_partial', _p(out), _p(table), M, V, d, passes, _p(part), _stream())
    return part


def ce_finalize(partial, out, table, target, n_groups, idx_offset=0):
    M, d = out.shape
    dev = out.device
    lse = torch.empty(M, dtype=torch.float32, device=dev)
    tgt = torch.empty_like(lse)
    row_loss = torch.empty_like(lse)
    loss = torch.empty(n_groups, dtype=torch.float32, device=dev)
    LIB.call('acsr_ce_finalize', _p(partial), partial.shape[1], _p(out), _p(table), _p(target, torch.int64), M, d,
             table.shape[0], idx_offset, n_groups, _p(lse), _p(tgt), _p(row_loss), _p(loss), _stream())
    return lse, tgt, row_loss, loss


def ce_grad_matrix_t(out, table, lse, target, row_scale, passes=3):
    """Gt [V, M] = ((softmax - onehot) * row_scale)^T  (transposed so the epilogue's stores coalesce)."""
    M, d = out.shape
    V = table.shape[0]
    Gt = torch.empty((V, M), dtype=torch.float32, device=out.device)
    LIB.call('acsr_logits_ce_grad', _p(out), _p(table), _p(lse), _p(target, torch.int64), _p(row_scale), M, V, d, passes,
             _p(Gt), M, _stream())
    return Gt


def ce_bwd_dout(out, table, lse, target, row_scale, d_out, passes=3):
    """d_out [M,64] += G . E with G = (softmax - onehot) * row_scale recomputed tile by tile and kept in registers
    (acsr_ce_bwd_dout, hidden size 64): no [M,V] gradient matrix."""
    M, d = out.shape
    LIB.call('acsr_ce_bwd_dout', _p(out), _p(table), _p(lse), _p(target, torch.int64), _p(row_scale), M, table.shape[0], d, passes,
             _p(d_out), _stream())
    return d_out


def ce_bwd_dtable(out, table, lse, target, row_scale, d_table, passes=3, stream=None):
    """d_table [V,64] += G^T . out (acsr_ce_bwd_dtable, hidden size 64); rows of `out` whose row_scale is 0 contribute nothing."""
    M, d = out.shape
    LIB.call('acsr_ce_bwd_dtable', _p(out), _p(table), _p(lse), _p(target, torch.int64), _p(row_scale), M, table.shape[0], d, passes,
             _p(d_table), _stream() if stream is None else stream)
    return d_table


def linear_wgrad(dY, X, dW=None, db=None, want_bias=True):
    """dW [N,K] += dY^T.X and db [N] += colsum(dY) with the token axis split over the GPU (acsr_linear_wgrad)."""
    N, K = dY.shape[-1], X.shape[-1]
    dY2, X2 = dY.reshape(-1, N), X.reshape(-1, K)
    if not dY2.is_contiguous():
        dY2 = dY2.contiguous()
    if not X2.is_contiguous():
        X2 = X2.contiguous()
    if dW is None:
        dW = torch.zeros((N, K), dtype=torch.float32, device=dY.device)
    if db is None and want_bias:
        db = torch.zeros(N, dtype=torch.float32, device=dY.device)
    LIB.call('acsr_linear_wgrad', _p(dY2), _p(X2), dY2.shape[0], N, K, _p(dW), _p(db), _stream())
    return dW, db


def linear_tc(X, rows, W, N, w_sn, w_sk, bias, Y, ldy, accumulate=False, batch=1, sx=0, sw=0, sb=0, sy=0, passes=3):
    """Y[rows,N] (+)= X[rows,64].Wt^T + bias on tcgen05 (acsr_linear_tc); pointers may be views, strides in floats."""
    LIB.call('acsr_linear_tc', _p(X), int(rows), 64, _p(W), int(N), int(w_sn), int(w_sk), _p(bias), int(bool(accumulate)),
             _p(Y), int(ldy), int(batch), int(sx), int(sw), int(sb), int(sy), passes, _stream())


def linear_tok(X, rows, K, W, N, Y, ldy, ldx=None, xkb=64, w_sn=None, w_sk=1, wkb=64, bias=None, accumulate=False,
               batch=1, sx=0, sw=0, sb=0, sy=0, passes=3):
    """Y[rows,N] (+)= X.W^T + bias on tcgen05 with token rows on the M axis (acsr_linear_tok); strides in floats."""
    LIB.call('acsr_linear_tok', _p(X), int(K if ldx is None else ldx), int(xkb), int(rows), int(K), _p(W),
             int(K if w_sn is None else w_sn), int(w_sk), int(wkb), int(N), _p(bias), int(bool(accumulate)), _p(Y), int(ldy),
             int(batch), int(sx), int(sw), int(sb), int(sy), passes, _stream())


def linear_tok_bdrl(X, rows, K, W, bias, res, res_rows, ln_w, ln_b, eps, p, mask, rngp, rng_stream, HZ, out, stats, passes=3):
    """HZ = X.W^T ; out = LN(dropout(HZ + bias) + res) ; stats = (mean, rstd)  (acsr_linear_tok_bdrl, width 64)."""
    LIB.call('acsr_linear_tok_bdrl', _p(X), int(K), int(rows), int(K), _p(W), _p(bias), _p(res), int(res_rows), _p(ln_w), _p(ln_b),
             float(eps), float(p), _p(mask), rngp, int(rng_stream), _p(HZ), _p(out), _p(stats), passes, _stream())


def _linear_grad_buffers(weight, bias):
    """(dW, db) destinations of a weight-gradient problem: both always exist (the kernel writes both), in place when possible"""
    sw, sb = _grad_sink(weight), (_grad_sink(bias) if bias is not None else None)
    if sw is not None and (bias is None or sb is not None):
        return (sw, sb), (None, None)
    dW = torch.zeros(weight.shape, dtype=torch.float32, device=weight.device)
    db = torch.zeros(bias.shape, dtype=torch.float32, device=weight.device) if bias is not None else None
    return (dW, db), (dW, db)


class LinearFn(torch.autograd.Function):
    """y = x.W^T (+ b) -- every nn.Linear of the API-compatible (autograd) path.  Forward, dX and dW/db all run on the
    K-streamed tcgen05 kernel (acsr_gemm_batch, 3xTF32): no library GEMM."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        ctx.bias_ref = bias
        N, K = weight.shape
        x2 = x.reshape(-1, K)
        if not x2.is_contiguous():
            x2 = x2.contiguous()
        w = weight if weight.is_contiguous() else weight.contiguous()
        y = torch.empty((x2.shape[0], N), dtype=torch.float32, device=x.device)
        gemm_batch([gemm_problem(x2, w, y, x2.shape[0], N, K, bias=bias)])
        return y.view(*x.shape[:-1], N)

    @staticmethod
    def backward(ctx, dy):
        x, weight = ctx.saved_tensors
        N, K = weight.shape
        dy2 = dy.reshape(-1, N)
        if not dy2.is_contiguous():
            dy2 = dy2.contiguous()
        rows = dy2.shape[0]
        dx = dW = db = None
        if ctx.needs_input_grad[0]:
            w = weight if weight.is_contiguous() else weight.contiguous()
            dx = torch.empty((rows, K), dtype=torch.float32, device=dy.device)
            gemm_batch([gemm_problem(dy2, w, dx, rows, K, N, b_strides=(1, K, 0, N))])      # dx = dy.W: weight read transposed
            dx = dx.view_as(x)
        if (ctx.needs_input_grad[1] and _wants_grad(weight)) or (ctx.has_bias and ctx.needs_input_grad[2] and _wants_grad(ctx.bias_ref)):
            x2 = x.reshape(-1, K)
            if not x2.is_contiguous():
                x2 = x2.contiguous()
            (bW, bb), (dW, db) = _linear_grad_buffers(weight, ctx.bias_ref)
            gemm_batch([wgrad_problem(dy2, x2, rows, N, K, bW, bb)])
        return dx, dW, db


def linear(x, weight, bias=None):
    return LinearFn.apply(x, weight, bias)


class MultiLinearFn(torch.autograd.Function):
    """n independent y_i = x_i.W_i^T (+ b_i) as ONE launch of the K-streamed tcgen05 GEMM (a problem list), and in the backward one
    launch for all input gradients and one for all weight / bias gradients -- the Q/K/V projections, the attack pair + gate,
    and the attacked / calibrated streams through the same dense or feed-forward weight (layers.py:658-659, 680, 687-689,
    791-794, 887).  Inputs / weights may repeat; autograd sums the returned gradients."""

    @staticmethod
    def forward(ctx, n, *args):
        xs, ws, bs = args[:n], args[n:2 * n], args[2 * n:3 * n]
        ctx.set_materialize_grads(False)
        x2s, ys, pr, keep = [], [], [], []
        for x, w, b in zip(xs, ws, bs):
            N, K = w.shape
            x2 = x.reshape(-1, K)
            x2 = x2 if x2.is_contiguous() else x2.contiguous()
            w = w if w.is_contiguous() else w.contiguous()
            keep.append(w)
            y = torch.empty((x2.shape[0], N), dtype=torch.float32, device=x.device)
            pr.append(gemm_problem(x2, w, y, x2.shape[0], N, K, bias=b))
            x2s.append(x2)
            ys.append(y.view(*x.shape[:-1], N))
        gemm_batch(pr)
        ctx.save_for_backward(*x2s, *ws)
        ctx.n, ctx.bias_refs, ctx.x_shapes = n, bs, [x.shape for x in xs]
        return tuple(ys)

    @staticmethod
    def backward(ctx, *dys):
        n = ctx.n
        saved = ctx.saved_tensors
        x2s, ws = saved[:n], saved[n:]
        dxs, dWs, dbs = [None] * n, [None] * n, [None] * n
        pr_x, pr_w = [], []
        keep = []          # every operand of a problem stays referenced until its launch (a freed temporary could be handed out again)
        for i, dy in enumerate(dys):
            if dy is None:
                continue
            w, b = ws[i], ctx.bias_refs[i]
            N, K = w.shape
            dy2 = dy.reshape(-1, N)
            dy2 = dy2 if dy2.is_contiguous() else dy2.contiguous()
            keep.append(dy2)
            rows = dy2.shape[0]
            if ctx.needs_input_grad[1 + i]:
                wc = w if w.is_contiguous() else w.contiguous()
                keep.append(wc)
                dx = torch.empty((rows, K), dtype=torch.float32, device=dy.device)
                pr_x.append(gemm_problem(dy2, wc, dx, rows, K, N, b_strides=(1, K, 0, N)))
                dxs[i] = dx.view(ctx.x_shapes[i])
            if (ctx.needs_input_grad[1 + n + i] and _wants_grad(w)) or (b is not None and ctx.needs_input_grad[1 + 2 * n + i] and _wants_grad(b)):
                (bW, bb), (dWs[i], dbs[i]) = _linear_grad_buffers(w, b)
                keep += [bW, bb]
                pr_w.append(wgrad_problem(dy2, x2s[i], rows, N, K, bW, bb))
        if pr_x:
            gemm_batch(pr_x)
        if pr_w:
            gemm_batch(pr_w)
        del keep
        return (None, *dxs, *dWs, *dbs)


def multi_linear(xs, weights, biases=None):
    """[x_i.W_i^T + b_i] as one launch (MultiLinearFn)"""
    n = len(xs)
    biases = list(biases) if biases is not None else [None] * n
    return MultiLinearFn.apply(n, *xs, *weights, *biases)


class GatherRowsFn(torch.autograd.Function):
    """rows x[idx] of a [T, d] matrix (AcBERT4Rec: the hidden states of the masked positions, acbert4rec.py:214-222 does it with a
    one-hot bmm); backward: scatter-add of the gradient rows."""

    @staticmethod
    def forward(ctx, x, idx):
        x = x.contiguous()
        T, d = x.shape
        ids = (idx.reshape(-1) + 1).contiguous()          # ids 1..T over a table whose first row is id 1: no id looks like padding
        out = torch.empty((ids.numel(), d), dtype=torch.float32, device=x.device)
        LIB.call('acsr_shard_gather_rows', _p(ids, torch.int64), ids.numel(), _p(x), 1, T + 1, d, _p(out), _stream())
        ctx.save_for_backward(ids)
        ctx.meta = (T, d)
        return out

    @staticmethod
    def backward(ctx, d_out):
        (ids,) = ctx.saved_tensors
        T, d = ctx.meta
        d_x = torch.zeros((T, d), dtype=torch.float32, device=d_out.device)
        LIB.call('acsr_shard_scatter_add_rows', _p(ids, torch.int64), ids.numel(), _p(d_out.contiguous()), 1, T + 1, d, _p(d_x), _stream())
        return d_x, None


class LogitsCEFn(torch.autograd.Function):
    """loss[g] = mean CE over row group g of softmax(out.E^T) vs target -- acsasrec.py:117-121.
    Logits never materialise, forward or backward: at hidden size 64 the backward recomputes the logits tile by tile on the
    tensor cores and consumes G = (softmax - onehot) * row_scale in registers (acsr_ce_bwd_dout / acsr_ce_bwd_dtable).  Other
    widths write Gt once, then d_E = Gt.out and d_out = Gt^T.E (reduction over the catalogue) as two problems of one tcgen05
    launch (acsr_gemm_batch)."""

    @staticmethod
    def forward(ctx, out, table, target, n_groups, passes, row_weight=None):
        """row_weight [M] (optional): loss[g] = sum(w * row_loss) / sum(w) over the group (AcBERT4Rec's masked-item CE,
        acbert4rec.py:198-205); default: the plain mean."""
        out, table, target = out.contiguous(), table.contiguous(), target.contiguous()
        part = ce_partial(out, table, passes)
        lse, _, row_loss, loss = ce_finalize(part, out, table, target, n_groups)
        wn = None
        if row_weight is not None:
            w = row_weight.to(torch.float32).view(n_groups, -1)
            wn = (w / w.sum(1, keepdim=True)).reshape(-1).contiguous()      # normalised weights: d loss[g] / d row_loss
            loss = (row_loss.view(n_groups, -1) * wn.view(n_groups, -1)).sum(1)
        ctx.save_for_backward(out, table, target, lse, wn)
        ctx.meta = (n_groups, passes)
        return loss

    @staticmethod
    def backward(ctx, d_loss):
        out, table, target, lse, wn = ctx.saved_tensors
        n_groups, passes = ctx.meta
        M = out.shape[0]
        per = M // n_groups
        if wn is not None:
            row_scale = (d_loss.to(torch.float32).view(n_groups, 1) * wn.view(n_groups, per)).reshape(-1).contiguous()
        else:
            row_scale = (d_loss.to(torch.float32) / per).view(n_groups, 1).expand(n_groups, per).reshape(-1).contiguous()
        V, d = table.shape
        d_out = d_table = None
        if d == 64:
            if ctx.needs_input_grad[0]:
                d_out = ce_bwd_dout(out, table, lse, target, row_scale, torch.zeros((M, d), dtype=torch.float32, device=out.device), passes)
            if ctx.needs_input_grad[1] and _wants_grad(table):
                d_table = ce_bwd_dtable(out, table, lse, target, row_scale, torch.zeros((V, d), dtype=torch.float32, device=out.device), passes)
            return d_out, d_table, None, None, None, None
        Gt = ce_grad_matrix_t(out, table, lse, target, row_scale, passes)
        pr = []
        if ctx.needs_input_grad[0]:            # d_out [M,d] = Gt^T . E : contraction over the catalogue, split over the CTAs
            d_out = torch.zeros((M, d), dtype=torch.float32, device=out.device)
            pr.append(wgrad_problem(Gt, table, V, M, d, d_out))
        if ctx.needs_input_grad[1] and _wants_grad(table):            # d_E [V,d] = Gt . out
            d_table = torch.empty((V, d), dtype=torch.float32, device=out.device)
            pr.append(gemm_problem(Gt, out, d_table, V, d, M, b_strides=(1, d, 0, M)))
        if pr:
            gemm_batch(pr)
        return d_out, d_table, None, None, None, None



class BprLossFn(torch.autograd.Function):
    """loss[g] = mean over row group g of -log(gamma + sigmoid(out.E[pos] - out.E[neg])) -- acsasrec.py:109-116, loss.py:21-47."""

    @staticmethod
    def forward(ctx, out, table, pos_items, neg_items, n_groups, gamma):
        out, table = out.contiguous(), table.contiguous()
        pos_items, neg_items = pos_items.contiguous(), neg_items.contiguous()
        M, d = out.shape
        dev = out.device
        row_x = torch.empty(M, dtype=torch.float32, device=dev)
        row_loss = torch.empty(M, dtype=torch.float32, device=dev)
        loss = torch.empty(n_groups, dtype=torch.float32, device=dev)
        LIB.call('acsr_bpr_loss_fwd', _p(out), _p(table), _p(pos_items, torch.int64), _p(neg_items, torch.int64), M, d, n_groups,
                 float(gamma), _p(row_x), _p(row_loss), _p(loss), _stream())
        ctx.save_for_backward(out, table, pos_items, neg_items, row_x)
        ctx.meta = (n_groups, float(gamma))
        return loss

    @staticmethod
    def backward(ctx, d_loss):
        out, table, pos_items, neg_items, row_x = ctx.saved_tensors
        n_groups, gamma = ctx.meta
        M, d = out.shape
        per = M // n_groups
        row_scale = (d_loss.to(torch.float32) / per).view(n_groups, 1).expand(n_groups, per).reshape(-1).contiguous()
        d_out = torch.empty_like(out) if ctx.needs_input_grad[0] else None
        d_table = torch.zeros_like(table) if ctx.needs_input_grad[1] else None
        LIB.call('acsr_bpr_loss_bwd', _p(out), _p(table), _p(pos_items, torch.int64), _p(neg_items, torch.int64), _p(row_x),
                 _p(row_scale), M, d, gamma, 0, M, _p(d_out), _p(d_table), _stream())
        return d_out, d_table, None, None, None, None


def bpr_dots_shard(out, shard, lo, hi, V, pos_items, neg_items):
    """dots [M, 2] = (out . E[pos], out . E[neg]) over the ids this rank owns (E[i] = shard[i - lo] for i in [lo, hi)), 0 for
    the others: summed over the ranks, BprLossFn's two scores bit for bit (acsr_bpr_dots_shard)"""
    out, pos_items, neg_items = out.contiguous(), pos_items.contiguous(), neg_items.contiguous()
    M, d = out.shape
    dots = torch.empty((M, 2), dtype=torch.float32, device=out.device)
    LIB.call('acsr_bpr_dots_shard', _p(out), _p(shard.contiguous()), int(lo), int(hi), int(V), _p(pos_items, torch.int64),
             _p(neg_items, torch.int64), M, d, _p(dots), _stream())
    return dots


def bpr_loss_from_dots(dots, n_groups, gamma):
    """summed dots [M, 2] -> (loss [n_groups], row_x [M]) as BprLossFn's forward computes them (acsr_bpr_loss_from_dots)"""
    dots = dots.contiguous()
    M = dots.shape[0]
    row_x = torch.empty(M, dtype=torch.float32, device=dots.device)
    row_loss = torch.empty(M, dtype=torch.float32, device=dots.device)
    loss = torch.empty(n_groups, dtype=torch.float32, device=dots.device)
    LIB.call('acsr_bpr_loss_from_dots', _p(dots), M, int(n_groups), float(gamma), _p(row_x), _p(row_loss), _p(loss), _stream())
    return loss, row_x


def bpr_loss_bwd_shard(out, shard, lo, hi, V, pos_items, neg_items, row_x, row_scale, gamma, table_row_begin=0, table_row_end=0,
                       shard_grad=None):
    """BprLossFn's backward over the ids this rank owns (acsr_bpr_loss_bwd_shard) -> d_out [M, d], this rank's part of
    g * (E[pos] - E[neg]); rows [table_row_begin, table_row_end) add +-g * out into shard_grad rows of owned ids"""
    out = out.contiguous()
    M, d = out.shape
    d_out = torch.empty_like(out)
    LIB.call('acsr_bpr_loss_bwd_shard', _p(out), _p(shard.contiguous()), int(lo), int(hi), int(V), _p(pos_items.contiguous(), torch.int64),
             _p(neg_items.contiguous(), torch.int64), _p(row_x.contiguous()), _p(row_scale.contiguous()), M, d, float(gamma),
             int(table_row_begin), int(table_row_end), _p(d_out), _p(shard_grad), _stream())
    return d_out


def logits_scores(out, table, passes=3):
    """scores [M,V] = out.E^T (contiguous)  -- acsasrec.py:162-163."""
    out, table = out.contiguous(), table.contiguous()
    M, d = out.shape
    V = table.shape[0]
    scores = torch.empty((M, V), dtype=torch.float32, device=out.device)
    LIB.call('acsr_logits_store', _p(out), _p(table), M, V, d, passes, _p(scores), V, _stream())
    return scores


def logits_topk_partial(out, table, k, idx_offset=0, skip_col0=True, passes=3, share_bound=True):
    out, table = out.contiguous(), table.contiguous()
    M, d = out.shape
    V = table.shape[0]
    nc = logits_num_chunks(M, V)
    pv = torch.empty((M, nc, k), dtype=torch.float32, device=out.device)
    pi = torch.empty((M, nc, k), dtype=torch.int64, device=out.device)
    # scratch for the per-row lower bound the CTAs of the launch share (acsr_logits_topk_partial_ws)
    rb = torch.empty(2 * M * nc, dtype=torch.int32, device=out.device) if share_bound else None
    LIB.call('acsr_logits_topk_partial_ws', _p(out), _p(table), M, V, d, passes, k, idx_offset, int(skip_col0),
             _p(pv), _p(pi, torch.int64), _p(rb, torch.int32), _stream())
    return pv, pi


def topk_merge(pv, pi, k, positive=None):
    """-> (val [M,k], idx [M,k] int64, rec_topk [M,k+1] int32 | None)."""
    M = pv.shape[0]
    pv = pv.reshape(M, -1, k).contiguous()
    pi = pi.reshape(M, -1, k).contiguous()
    dev = pv.device
    val = torch.empty((M, k), dtype=torch.float32, device=dev)
    idx = torch.empty((M, k), dtype=torch.int64, device=dev)
    rec = torch.empty((M, k + 1), dtype=torch.int32, device=dev) if positive is not None else None
    LIB.call('acsr_topk_merge', _p(pv), _p(pi, torch.int64), M, pv.shape[1], k,
             _p(positive.contiguous(), torch.int64) if positive is not None else None,
             _p(val), _p(idx, torch.int64), _p(rec, torch.int32), _stream())
    return val, idx, rec


def topk_select(scores, k, positive=None, skip_col0=True, idx_offset=0):
    """row-wise top-k of a dense score matrix (radix select in shared memory) -> (val, idx, rec_topk | None)."""
    M, V = scores.shape
    dev = scores.device
    if not scores.is_cuda or scores.dtype != torch.float32 or scores.stride(1) != 1:
        raise AcsrError('topk_select: scores must be a float32 CUDA matrix with unit column stride (rows may be strided)')
    val = torch.empty((M, k), dtype=torch.float32, device=dev)
    idx = torch.empty((M, k), dtype=torch.int64, device=dev)
    rec = torch.empty((M, k + 1), dtype=torch.int32, device=dev) if positive is not None else None
    LIB.call('acsr_topk_select', scores.data_ptr(), M, V, scores.stride(0), k, int(skip_col0), idx_offset,
             _p(positive.contiguous(), torch.int64) if positive is not None else None,
             _p(val), _p(idx, torch.int64), _p(rec, torch.int32), _stream())
    return val, idx, rec


def _check_positive(positive, M, who):
    if positive is None or positive.dim() != 1 or positive.shape[0] != M:
        raise AcsrError('%s: positive must be a 1-D tensor of %d item ids (got %s)' % (who, M, None if positive is None else tuple(positive.shape)))
    return positive.contiguous()


def row_dot(out, table, ids, idx_offset=0):
    """dot [M] = out[m] . table[ids[m] - idx_offset] in fp32 (0 where that row is not in this table / shard), the positive's score
    the rank counts are taken against (acsr_row_dot)"""
    out, table = out.contiguous(), table.contiguous()
    M, d = out.shape
    if table.dim() != 2 or table.shape[1] != d:
        raise AcsrError('row_dot: out %s and table %s disagree' % (tuple(out.shape), tuple(table.shape)))
    ids = _check_positive(ids, M, 'row_dot')
    dot = torch.empty(M, dtype=torch.float32, device=out.device)
    LIB.call('acsr_row_dot', _p(out), _p(table), _p(ids, torch.int64), M, d, table.shape[0], int(idx_offset), _p(dot), _stream())
    return dot


def logits_topk_rank_partial(out, table, k, positive, pos_score, idx_offset=0, skip_col0=True, passes=3, share_bound=True):
    """logits_topk_partial + per-(row, chunk) counts [M, nc, 2] int32 of the scores above / equal to pos_score (GAUC)"""
    out, table = out.contiguous(), table.contiguous()
    M, d = out.shape
    V = table.shape[0]
    positive = _check_positive(positive, M, 'logits_topk_rank_partial')
    if pos_score.shape != (M,):
        raise AcsrError('logits_topk_rank_partial: pos_score must be [%d] (got %s)' % (M, tuple(pos_score.shape)))
    nc = logits_num_chunks(M, V)
    pv = torch.empty((M, nc, k), dtype=torch.float32, device=out.device)
    pi = torch.empty((M, nc, k), dtype=torch.int64, device=out.device)
    pc = torch.empty((M, nc, 2), dtype=torch.int32, device=out.device)
    rb = torch.empty(2 * M * nc, dtype=torch.int32, device=out.device) if share_bound else None
    LIB.call('acsr_logits_topk_rank_partial', _p(out), _p(table), M, V, d, passes, k, idx_offset, int(skip_col0),
             _p(positive, torch.int64), _p(pos_score.contiguous()), _p(pv), _p(pi, torch.int64), _p(pc, torch.int32),
             _p(rb, torch.int32), _stream())
    return pv, pi, pc


def topk_merge_rank(pv, pi, k, pc, positive=None):
    """topk_merge + the sum of the per-part counts pc [M, n, 2] -> (val, idx, rec | None, counts [M, 2] int32)"""
    M = pv.shape[0]
    pv = pv.reshape(M, -1, k).contiguous()
    pi = pi.reshape(M, -1, k).contiguous()
    pc = pc.reshape(M, -1, 2).contiguous()
    dev = pv.device
    val = torch.empty((M, k), dtype=torch.float32, device=dev)
    idx = torch.empty((M, k), dtype=torch.int64, device=dev)
    rec = torch.empty((M, k + 1), dtype=torch.int32, device=dev) if positive is not None else None
    counts = torch.empty((M, 2), dtype=torch.int32, device=dev)
    LIB.call('acsr_topk_merge_rank', _p(pv), _p(pi, torch.int64), M, pv.shape[1], k,
             _p(positive.contiguous(), torch.int64) if positive is not None else None, _p(pc, torch.int32), pc.shape[1],
             _p(val), _p(idx, torch.int64), _p(rec, torch.int32), _p(counts, torch.int32), _stream())
    return val, idx, rec, counts


def topk_select_rank(scores, k, positive, pos_score, skip_col0=True, idx_offset=0):
    """topk_select + counts [M, 2] int32 of the row's scores above / equal to pos_score (the positive's column left out)"""
    M, V = scores.shape
    dev = scores.device
    if not scores.is_cuda or scores.dtype != torch.float32 or scores.stride(1) != 1:
        raise AcsrError('topk_select_rank: scores must be a float32 CUDA matrix with unit column stride (rows may be strided)')
    positive = _check_positive(positive, M, 'topk_select_rank')
    val = torch.empty((M, k), dtype=torch.float32, device=dev)
    idx = torch.empty((M, k), dtype=torch.int64, device=dev)
    rec = torch.empty((M, k + 1), dtype=torch.int32, device=dev)
    counts = torch.empty((M, 2), dtype=torch.int32, device=dev)
    LIB.call('acsr_topk_select_rank', scores.data_ptr(), M, V, scores.stride(0), k, int(skip_col0), idx_offset,
             _p(positive, torch.int64), _p(pos_score.contiguous()), _p(val), _p(idx, torch.int64), _p(rec, torch.int32),
             _p(counts, torch.int32), _stream())
    return val, idx, rec, counts


_SELECT_MAX = []


def full_sort_topk(out, table, k, positive=None, passes=3, counts=False):
    """scores -> scores[:,0]=-inf -> top-k -> hit flags (trainer.py:941-942, collector.py:147-153).  Small catalogues
    (one row of scores fits in shared memory): tensor-core scores, L2-resident, + radix select; large ones: the fused
    logits + streaming top-k kernel and a merge of its per-chunk lists (the scores never exist).
    counts=True (needs positive): also -> counts [M, 2] int32 = (#items scoring above, #items tied with) the positive's fp32 score
    (row_dot), column 0 and the positive itself not counted -- GAUC's average rank without sorting the catalogue."""
    if not _SELECT_MAX:
        _SELECT_MAX.append(LIB.query('acsr_topk_select_max_items'))
    V = table.shape[0]
    if counts:
        s_pos = row_dot(out, table, _check_positive(positive, out.shape[0], 'full_sort_topk'))
        if V <= _SELECT_MAX[0] and V - 1 >= k:
            return topk_select_rank(logits_scores(out, table, passes), k, positive, s_pos)
        pv, pi, pc = logits_topk_rank_partial(out, table, k, positive, s_pos, 0, True, passes)
        return topk_merge_rank(pv, pi, k, pc, positive)
    if V <= _SELECT_MAX[0] and V - 1 >= k:
        return topk_select(logits_scores(out, table, passes), k, positive)
    pv, pi = logits_topk_partial(out, table, k, 0, True, passes)
    return topk_merge(pv, pi, k, positive)


# ------------------------------------------------------------------------------------------
# negative sampling and sampled-candidate ranking (negsample.cu)
# ------------------------------------------------------------------------------------------
def neg_sample(users, n_neg, used_offsets, used_items, n_items, rng, rng_stream, positives=None, alias=None, out=None, ld=None,
               perm=None, cursor=None, n_rows=0, rows=None):
    """-> negs [M, n_neg] int64: per row, items of [1, n_items) outside the user's used set (acsr_neg_sample).  out may be a
    row-strided view (ld = its row stride, e.g. columns 1.. of a candidate matrix).  With perm / cursor, row m reads users /
    positives at perm[cursor * rows + m] (the batch acsr_batch_gather writes)."""
    M = int(rows if rows is not None else users.shape[0])
    n_src = int(n_rows) if perm is not None else M                   # rows users / positives are read at
    if users.dim() != 1 or users.shape[0] < n_src or (positives is not None and tuple(positives.shape) != tuple(users.shape)):
        raise AcsrError('neg_sample: users (and positives) must be 1-D with at least %d rows (got %s)' % (n_src, tuple(users.shape)))
    if perm is not None and perm.numel() != n_src:
        raise AcsrError('neg_sample: perm has %d entries, n_rows is %d' % (perm.numel(), n_src))
    if out is None:
        out = torch.empty((M, n_neg), dtype=torch.int64, device=used_items.device)
        ld = n_neg
    if out.dim() != 2 or tuple(out.shape) != (M, int(n_neg)):
        raise AcsrError('neg_sample: out must be a [%d, %d] matrix (got %s)' % (M, n_neg, tuple(out.shape)))
    if ld is None:
        ld = out.stride(0)
    if not out.is_cuda or out.dtype != torch.int64 or out.stride(1) != 1 or (M > 1 and out.stride(0) != ld) or ld < n_neg:
        raise AcsrError('neg_sample: out must be an int64 CUDA matrix with unit column stride and row stride ld >= n_neg')
    prob, idx = alias if alias is not None else (None, None)
    LIB.call('acsr_neg_sample', _p(users, torch.int64), _p(positives, torch.int64), _p(perm, torch.int64), _p(cursor, torch.int64),
             int(n_rows), M, int(n_neg), _p(used_offsets, torch.int64), _p(used_items, torch.int64), used_offsets.numel() - 1,
             int(n_items), _p(prob), _p(idx, torch.int64), rng.ptr, int(rng_stream), out.data_ptr(), int(ld), _stream())
    return out


def candidate_rank(out, table, cand, k, want_scores=False, want_counts=False):
    """rank of column 0 of cand [M, 1+N] among the distinct other candidates by out[m] . table[c] (fp32), as the hit-flag
    matrix rec [M, k+1] int32 of the evaluator (acsr_candidate_rank) -> (rec, scores [M, 1+N] | None); want_counts: -> (rec,
    scores | None, counts [M, 3] int32 = distinct negatives above / tied with the positive, distinct candidates)"""
    out, table, cand = out.contiguous(), table.contiguous(), cand.contiguous()
    if out.dim() != 2 or table.dim() != 2 or cand.dim() != 2:
        raise AcsrError('candidate_rank: out [M, d], table [V, d] and cand [M, 1+N] must be matrices')
    M, d = out.shape
    if table.shape[1] != d or cand.shape[0] != M or int(k) < 1:
        raise AcsrError('candidate_rank: out %s, table %s and cand %s disagree (or k=%d < 1)' % (tuple(out.shape), tuple(table.shape),
                                                                                            tuple(cand.shape), int(k)))
    rec = torch.empty((M, k + 1), dtype=torch.int32, device=out.device)
    scores = torch.empty(cand.shape, dtype=torch.float32, device=out.device) if want_scores else None
    if want_counts:
        counts = torch.empty((M, 3), dtype=torch.int32, device=out.device)
        LIB.call('acsr_candidate_rank_counts', _p(out), _p(table), table.shape[0], d, _p(cand, torch.int64), M, cand.shape[1], int(k),
                 _p(rec, torch.int32), _p(scores), _p(counts, torch.int32), _stream())
        return rec, scores, counts
    LIB.call('acsr_candidate_rank', _p(out), _p(table), table.shape[0], d, _p(cand, torch.int64), M, cand.shape[1], int(k),
             _p(rec, torch.int32), _p(scores), _stream())
    return rec, scores


def candidate_scores_shard(out, shard, lo, hi, V, cand):
    """scores [M, 1+N] = out[m] . shard[id - lo] for the candidate ids (clamped to [0, V)) this rank owns, 0 for the others:
    the sum over the ranks is candidate_rank's scores bit for bit (acsr_candidate_scores_shard)"""
    out, cand = out.contiguous(), cand.contiguous()
    if out.dim() != 2 or shard.dim() != 2 or cand.dim() != 2 or shard.shape[1] != out.shape[1] or cand.shape[0] != out.shape[0]:
        raise AcsrError('candidate_scores_shard: out [M, d], shard [rows, d] and cand [M, 1+N] disagree (%s, %s, %s)'
                        % (tuple(out.shape), tuple(shard.shape), tuple(cand.shape)))
    if int(hi) - int(lo) > shard.shape[0]:
        raise AcsrError('candidate_scores_shard: rows [%d, %d) exceed the %d rows of the shard' % (int(lo), int(hi), shard.shape[0]))
    M, d = out.shape
    scores = torch.empty(cand.shape, dtype=torch.float32, device=out.device)
    LIB.call('acsr_candidate_scores_shard', _p(out), _p(shard.contiguous()), int(lo), int(hi), int(V), d, _p(cand, torch.int64), M,
             cand.shape[1], _p(scores), _stream())
    return scores


def candidate_rank_scores(scores, cand, V, k, want_counts=False):
    """candidate_rank's ranking of precomputed scores [M, 1+N] (acsr_candidate_rank_scores) -> (rec [M, k+1] int32, counts
    [M, 3] int32 | None)"""
    scores, cand = scores.contiguous(), cand.contiguous()
    if scores.dtype != torch.float32 or scores.dim() != 2 or tuple(cand.shape) != tuple(scores.shape) or int(k) < 1:
        raise AcsrError('candidate_rank_scores: float32 scores %s and cand %s must have one shape (and k=%d >= 1)'
                        % (tuple(scores.shape), tuple(cand.shape), int(k)))
    M = scores.shape[0]
    rec = torch.empty((M, k + 1), dtype=torch.int32, device=scores.device)
    counts = torch.empty((M, 3), dtype=torch.int32, device=scores.device) if want_counts else None
    LIB.call('acsr_candidate_rank_scores', _p(scores), _p(cand, torch.int64), int(V), M, scores.shape[1], int(k), _p(rec, torch.int32),
             _p(counts, torch.int32), _stream())
    return rec, counts


def used_item_csr(uid, iid, n_users, n_items):
    """per-user sorted unique items as a CSR (offsets [n_users+1], items) from parallel id arrays"""
    uid, iid = np.asarray(uid, dtype=np.int64), np.asarray(iid, dtype=np.int64)
    key = np.unique(uid * int(n_items) + iid)
    users, items = key // int(n_items), key % int(n_items)
    offsets = np.zeros(int(n_users) + 1, dtype=np.int64)
    np.cumsum(np.bincount(users, minlength=int(n_users)), out=offsets[1:])
    return offsets, items.astype(np.int64)


def alias_table(counts):
    """Walker alias table of the distribution counts / counts.sum() -> (prob float32, alias int64): draw i uniform, u uniform on
    (0, 1]; the item is i when u <= prob[i], else alias[i].  Vose's pairing, vectorised: the smalls (scaled mass < 1) are poured
    in order into the larges in order, so small i goes to the large whose cumulative excess E first reaches the smalls'
    cumulative deficit D before it, and large j, once D passes E_j, keeps 1 + E_j - D (its overflow) and aliases large j + 1."""
    w = np.asarray(counts, dtype=np.float64)
    n = len(w)
    scaled = w * (n / w.sum())
    prob = np.ones(n, dtype=np.float64)
    alias = np.arange(n, dtype=np.int64)
    small, large = np.nonzero(scaled < 1.0)[0], np.nonzero(scaled >= 1.0)[0]
    if len(small) and len(large):
        D = np.cumsum(1.0 - scaled[small])
        E = np.cumsum(scaled[large] - 1.0)
        j = np.searchsorted(E, np.concatenate(([0.0], D[:-1])), side='left')     # the large each small is poured into
        ok = j < len(large)                                                    # (beyond the last: rounding leftovers, kept ~1)
        prob[small[ok]], alias[small[ok]] = scaled[small[ok]], large[j[ok]]
        i = np.searchsorted(D, E, side='right')                                # the small whose deficit overflows large j
        sw = np.nonzero((i < len(small)) & (np.arange(len(large)) + 1 < len(large)))[0]
        prob[large[sw]], alias[large[sw]] = 1.0 + E[sw] - D[i[sw]], large[sw + 1]
    return prob.astype(np.float32), alias


class NegSampler(object):
    """Device-side negative sampler of one phase (RecBole 1.0.1's non-repeatable Sampler, sampler.py): the users' used sets as
    a CSR, for popularity the alias table of the item counts, and its own Philox state {seed, step} -- a DeviceRng separate
    from the model's dropout stream, so drawing negatives leaves training randomness untouched.  Every draw() advances the
    state first: each training step and each evaluation batch gets fresh negatives, reproducible from the seed."""

    RNG_STREAM = 0x4E470000                       # + phase: train / valid / test draw from disjoint counters

    def __init__(self, distribution, used_offsets, used_items, n_items, seed, phase=0, counts=None, alias=None):
        if distribution not in ('uniform', 'popularity'):
            raise ValueError('negative sampling distribution must be uniform or popularity (got %r)' % (distribution,))
        self.distribution, self.n_items, self.seed = distribution, int(n_items), int(seed)
        self.used_offsets, self.used_items = np.asarray(used_offsets, np.int64), np.asarray(used_items, np.int64)
        self.n_users = len(self.used_offsets) - 1
        self.rng_stream = self.RNG_STREAM + int(phase)
        self.alias = None
        if distribution == 'popularity':
            counts = np.asarray(counts, dtype=np.float64)
            if counts.shape != (self.n_items,) or counts.sum() <= 0:
                raise ValueError('popularity sampling needs item counts of shape [n_items] with a positive sum')
            self.counts = counts
            self.alias = alias if alias is not None else alias_table(counts)      # phases of one dataset share one table
        full = np.diff(self.used_offsets) >= self.n_items - 1
        if full.any():
            raise ValueError('user %d has interacted with every item: no negative can be drawn' % int(np.nonzero(full)[0][0]))
        self.rng = None
        self._dev = None

    def check_users(self, user_ids):
        """a row whose user id lies outside [0, n_users) gets item 0 from acsr_neg_sample: loaders reject such data up front"""
        u = np.asarray(user_ids.cpu() if torch.is_tensor(user_ids) else user_ids)
        if u.size and (u.min() < 0 or u.max() >= self.n_users):
            raise ValueError('user ids must lie in [0, %d) for this sampler (got %d..%d)' % (self.n_users, int(u.min()), int(u.max())))

    def to_device(self, device):
        """upload once per device ('cuda' and 'cuda:<current>' are the same device: the state a captured graph points at must
        not be replaced)"""
        device = torch.device(device)
        if device.type == 'cuda' and device.index is None:
            device = torch.device('cuda', torch.cuda.current_device())
        if self._dev is None or self._dev[0].device != device:
            t = [torch.from_numpy(self.used_offsets).to(device), torch.from_numpy(self.used_items).to(device)]
            if self.alias is not None:
                t += [torch.from_numpy(self.alias[0]).to(device), torch.from_numpy(self.alias[1]).to(device)]
            self._dev = t
            self.rng = DeviceRng(self.seed, device)
        return self

    def draw(self, users, n_neg, positives=None, out=None, ld=None, perm=None, cursor=None, n_rows=0, rows=None, advance=True):
        """advance the sampler's state (unless advance=False), then enqueue acsr_neg_sample -> negs [M, n_neg]"""
        self.to_device(users.device)
        if advance:
            self.rng.advance()
        alias = (self._dev[2], self._dev[3]) if self.alias is not None else None
        return neg_sample(users, n_neg, self._dev[0], self._dev[1], self.n_items, self.rng, self.rng_stream, positives, alias,
                          out, ld, perm, cursor, n_rows, rows)


def adam_step(param, grad, exp_avg, exp_avg_sq, step_count, lr, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.0):
    LIB.call('acsr_adam_step', _p(param), _p(grad), _p(exp_avg), _p(exp_avg_sq), param.numel(), lr, beta1, beta2, eps,
             weight_decay, _p(step_count, torch.int64), _stream())


def grad_norm_work(device):
    """scratch of grad_norm_partial: (per-CTA partials, arrival counter).  The counter starts at zero and the kernel leaves it
    at zero; launches that share one work pair must run in stream order."""
    return (torch.empty(LIB.query('acsr_grad_norm_max_blocks'), dtype=torch.float64, device=device),
            torch.zeros(1, dtype=torch.int32, device=device))


def grad_norm_partial(grad, norm_type, ranges=None, out=None, work=None):
    """acsr_grad_norm_partial -> out [1] float64: the sum of |g|^q over grad[begin:end] for every (begin, end) in ranges (default:
    all of grad), or max |g| for q = norm_type = inf.  acsr_adam_step_clipped combines such partials into the total norm."""
    ranges = [(0, grad.numel())] if ranges is None else [(int(b), int(e)) for b, e in ranges]
    rg = (ctypes.c_int64 * (2 * len(ranges)))(*[x for r in ranges for x in r])
    out = torch.empty(1, dtype=torch.float64, device=grad.device) if out is None else out
    work = grad_norm_work(grad.device) if work is None else work
    LIB.call('acsr_grad_norm_partial', _p(grad), grad.numel(), rg, len(ranges), float(norm_type), _p(work[0], torch.float64),
             _p(work[1], torch.int32), _p(out, torch.float64), _stream())
    return out


def adam_step_clipped(param, grad, exp_avg, exp_avg_sq, step_count, lr, partials, norm_type, max_norm, beta1=0.9, beta2=0.999,
                      eps=1e-8, weight_decay=0.0, total=None):
    """acsr_adam_step_clipped: clip_grad_norm_(max_norm, norm_type) with the total norm combined from `partials` (float64 [n],
    grad_norm_partial results of disjoint ranges, summed in index order), then adam_step on the clipped gradient, which is
    also written back to grad.  -> total [1] float32, the norm clip_grad_norm_ returns."""
    total = torch.empty(1, dtype=torch.float32, device=param.device) if total is None else total
    LIB.call('acsr_adam_step_clipped', _p(param), _p(grad), _p(exp_avg), _p(exp_avg_sq), param.numel(), lr, beta1, beta2, eps,
             weight_decay, _p(step_count, torch.int64), _p(partials, torch.float64), partials.numel(), float(norm_type),
             float(max_norm), _p(total), _stream())
    return total


# ------------------------------------------------------------------------------------------
# general tcgen05 GEMM (gemm_ks.cu): any hidden size, strided / transposed operands, problem lists
# ------------------------------------------------------------------------------------------
from ._lib import GemmProblem, EPI_STORE, EPI_ATOMIC, EPI_ACT, EPI_BDRL, GEMM_MAX_PROBLEMS  # noqa: E402


def gemm_problem(A, B, C, M, N, K, a_strides=None, b_strides=None, ldc=None, bias=None, epilogue=EPI_STORE, accumulate=False,
                 k_splits=0, colsum=None, act=0, C2=None, res=None, res_rows=0, ln_w=None, ln_b=None, eps=0.0, p_drop=0.0,
                 mask=None, rngp=None, rng_stream=0, out=None, stats=None):
    """one problem C[M,N] (+)= A[M,K].B[N,K]^T of an acsr_gemm_batch launch.  A / B / C are tensors (their data_ptr is the
    base address; views are fine) and a_strides / b_strides = (row_stride, k_stride, kblock_stride, kblock_len) in floats
    (default: row-major [rows, K]).  The caller keeps the tensors alive until the launch has been enqueued."""
    for t in (A, B, C, bias, colsum, C2, res, ln_w, ln_b, mask, out, stats):
        if t is not None and (not t.is_cuda or t.dtype != torch.float32):
            raise AcsrError('gemm_problem: float32 CUDA tensors only (no CPU fallback)')
    g = GemmProblem()
    ar, ak, akb, akl = a_strides if a_strides is not None else (K, 1, 0, K)
    br, bk, bkb, bkl = b_strides if b_strides is not None else (K, 1, 0, K)
    g.A, g.a_row_stride, g.a_k_stride, g.a_kb_stride, g.a_kblk = A.data_ptr(), int(ar), int(ak), int(akb), int(akl)
    g.B, g.b_row_stride, g.b_k_stride, g.b_kb_stride, g.b_kblk = B.data_ptr(), int(br), int(bk), int(bkb), int(bkl)
    g.C = C.data_ptr() if C is not None else None
    g.ldc = int(N if ldc is None else ldc)
    g.M, g.N, g.K = int(M), int(N), int(K)
    g.bias = bias.data_ptr() if bias is not None else None
    g.colsum = colsum.data_ptr() if colsum is not None else None
    g.C2 = C2.data_ptr() if C2 is not None else None
    g.res = res.data_ptr() if res is not None else None
    g.res_rows = int(res_rows)
    g.ln_w = ln_w.data_ptr() if ln_w is not None else None
    g.ln_b = ln_b.data_ptr() if ln_b is not None else None
    g.mask = mask.data_ptr() if mask is not None else None
    g.rng = rngp
    g.out = out.data_ptr() if out is not None else None
    g.stats = stats.data_ptr() if stats is not None else None
    g.epilogue, g.accumulate, g.k_splits, g.act = int(epilogue), int(bool(accumulate)), int(k_splits), int(act)
    g.rng_stream, g.eps, g.p_drop = int(rng_stream), float(eps), float(p_drop)
    return g


def gemm_batch(problems, passes=3, stream=None):
    """launch a list of gemm_problem()s (chunks of 16 per launch) on `stream` (default: the current torch stream)."""
    st = _stream() if stream is None else stream
    for i in range(0, len(problems), GEMM_MAX_PROBLEMS):
        chunk = problems[i:i + GEMM_MAX_PROBLEMS]
        arr = (GemmProblem * len(chunk))(*chunk)
        LIB.call('acsr_gemm_batch', arr, len(chunk), int(passes), st)


def wgrad_problem(dY, X, rows, N, K, dW, db=None, ldy=None, ldx=None, ldw=None, k_splits=0):
    """dW[N,K] += dY[:rows, :N]^T . X[:rows, :K]  (+ db[N] += column sums of dY): the token axis is the contraction."""
    ldy = N if ldy is None else ldy
    ldx = K if ldx is None else ldx
    return gemm_problem(dY, X, dW, N, K, rows, a_strides=(1, ldy, 0, rows), b_strides=(1, ldx, 0, rows), ldc=(K if ldw is None else ldw),
                        epilogue=EPI_ATOMIC, colsum=db, k_splits=k_splits)
