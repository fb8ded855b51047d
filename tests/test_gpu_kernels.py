"""Parity of every CUDA kernel (called through the C ABI via ops.py) against the CPU oracle on the
same seeded inputs.  Tolerances: fp32 arithmetic with a different summation order -> 2e-5 relative
to the tensor's max |value| for activations, 2e-4 for gradients (north_star: 1e-3)."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import acsr_oracle as O


@pytest.fixture(scope='module')
def A():
    import ac_tsr_b200 as pkg
    pkg.LIB.load()
    return pkg


def dev(t):
    return None if t is None else t.cuda()


def close(a, b, rtol, what=''):
    a = a.detach().double().cpu()
    b = b.detach().double().cpu()
    scale = float(b.abs().max().clamp(min=1e-30))
    err = float((a - b).abs().max())
    assert err <= rtol * scale + 1e-12, '%s: err %.3e scale %.3e' % (what, err, scale)


def drop(shape, p, g):
    return (torch.rand(shape, generator=g) >= p).float() / (1 - p)


# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize('d,use_pos,p', [(64, False, 0.5), (64, True, 0.0), (128, True, 0.5), (32, False, 0.2), (256, False, 0.5)])
def test_embed_ln_dropout(A, d, use_pos, p):
    g = torch.Generator().manual_seed(d + int(p * 10))
    B, L, V = 7, 50, 97
    seq, ln, _ = O.synth_batch(B, L, V, seed=3)
    E = torch.randn(V, d, generator=g) * 0.5
    pos = torch.randn(L, d, generator=g) * 0.3 if use_pos else None
    w = 1 + 0.1 * torch.randn(d, generator=g)
    b = 0.1 * torch.randn(d, generator=g)
    mask = drop((B, L, d), p, g) if p > 0 else None
    dy = torch.randn(B, L, d, generator=g)
    # oracle
    Eo, wo, bo = (t.clone().requires_grad_(True) for t in (E, w, b))
    po = pos.clone().requires_grad_(True) if use_pos else None
    yo = O.embed_ln_dropout(seq, Eo, wo, bo, 1e-12, O.Rand({'emb': mask} if mask is not None else {}), po)
    yo.backward(dy)
    # CUDA
    Ec, wc, bc = (t.clone().cuda().requires_grad_(True) for t in (E, w, b))
    pc = pos.clone().cuda().requires_grad_(True) if use_pos else None
    y = A.ops.EmbedLnDropoutFn.apply(seq.cuda(), Ec, pc, wc, bc, 1e-12, p, dev(mask), None, 1)
    close(y, yo, 2e-5, 'fwd')
    y.backward(dy.cuda())
    gE_ref = Eo.grad
    assert float(Ec.grad[0].abs().max()) == 0.0          # nn.Embedding(padding_idx=0)
    close(Ec.grad, gE_ref, 2e-4, 'dE')
    close(wc.grad, wo.grad, 2e-4, 'dw')
    close(bc.grad, bo.grad, 2e-4, 'db')
    if use_pos:
        close(pc.grad, po.grad, 2e-4, 'dpos')


@pytest.mark.parametrize('d,p,bias', [(64, 0.5, True), (64, 0.0, False), (128, 0.3, True), (256, 0.5, True)])
def test_bias_dropout_res_ln(A, d, p, bias):
    g = torch.Generator().manual_seed(5 + d)
    T = 333
    h, res = torch.randn(T, d, generator=g), torch.randn(T, d, generator=g)
    bi = torch.randn(d, generator=g) * 0.2 if bias else None
    w, b = 1 + 0.1 * torch.randn(d, generator=g), 0.1 * torch.randn(d, generator=g)
    mask = drop((T, d), p, g) if p > 0 else None
    dy = torch.randn(T, d, generator=g)
    ho, ro, wo, bo = (t.clone().requires_grad_(True) for t in (h, res, w, b))
    bio = bi.clone().requires_grad_(True) if bias else None
    z = ho + bio if bias else ho
    if mask is not None:
        z = z * mask
    yo = O.layer_norm(z + ro, wo, bo, 1e-12)
    yo.backward(dy)
    hc, rc, wc, bc = (t.clone().cuda().requires_grad_(True) for t in (h, res, w, b))
    bic = bi.clone().cuda().requires_grad_(True) if bias else None
    y = A.ops.BiasDropoutResLnFn.apply(hc, bic, rc, wc, bc, 1e-12, p, dev(mask), None, 0)
    close(y, yo, 2e-5, 'fwd')
    y.backward(dy.cuda())
    close(hc.grad, ho.grad, 2e-4, 'dh')
    close(rc.grad, ro.grad, 2e-4, 'dres')
    close(wc.grad, wo.grad, 2e-4, 'dw')
    close(bc.grad, bo.grad, 2e-4, 'db')
    if bias:
        close(bic.grad, bio.grad, 2e-4, 'dbias')


@pytest.mark.parametrize('act', ['gelu', 'relu', 'swish', 'tanh', 'sigmoid'])
@pytest.mark.parametrize('n', [64, 128, 256, 1024])
def test_bias_act(A, act, n):
    g = torch.Generator().manual_seed(n)
    T = 211
    h, b, dy = torch.randn(T, n, generator=g) * 2, torch.randn(n, generator=g), torch.randn(T, n, generator=g)
    ho, bo = h.clone().requires_grad_(True), b.clone().requires_grad_(True)
    yo = O.act_fn(act)(ho + bo)
    yo.backward(dy)
    hc, bc = h.clone().cuda().requires_grad_(True), b.clone().cuda().requires_grad_(True)
    y = A.ops.BiasActFn.apply(hc, bc, A.ops.ACT_IDS[act])
    close(y, yo, 1e-5, 'fwd')
    y.backward(dy.cuda())
    close(hc.grad, ho.grad, 2e-5, 'dh')
    close(bc.grad, bo.grad, 2e-4, 'dbias')


@pytest.mark.parametrize('B,L,I,groups,act,p', [(37, 7, 256, 2, 'gelu', 0.3), (256, 50, 256, 2, 'gelu', 0.5), (5, 50, 64, 1, 'relu', 0.0),
                                                (130, 20, 48, 2, 'swish', 0.2)])
def test_tail_fused_last_layer(A, B, L, I, groups, act, p):
    """acsr_tail_fwd / acsr_tail_bwd (the last layer's dense part on the rows that feed the losses, one launch per direction)
    against fp64 autograd of the same chain (layers.py:676-684, 790-798 + gather_indexes) with injected dropout masks."""
    from ac_tsr_b200._lib import LIB
    _p = A.ops._p
    g = torch.Generator().manual_seed(B * 3 + L + I)
    T, d, C = B * L, 64, groups * B
    r = lambda *s: torch.randn(*s, generator=g)       # noqa: E731
    ctx = [r(T, d) for _ in range(groups)]
    x = r(T, d)
    ln = torch.randint(1, L + 1, (B,), generator=g)
    ln[0] = 1
    ln[-1] = L
    Wo, bo, W1, b1, W2, b2 = r(d, d) * 0.2, r(d) * 0.1, r(I, d) * 0.2, r(I) * 0.1, r(d, I) * 0.1, r(d) * 0.1
    lnAw, lnAb, lnFw, lnFb = 1 + 0.1 * r(d), 0.1 * r(d), 1 + 0.1 * r(d), 0.1 * r(d)
    m_a, m_f = drop((C, d), p, g), drop((C, d), p, g)
    d_out = r(C, d)
    # ---- fp64 reference ----
    P = [t.double().requires_grad_(True) for t in (Wo, bo, W1, b1, W2, b2, lnAw, lnAb, lnFw, lnFb)]
    cd = [t.double().requires_grad_(True) for t in ctx]
    xd = x.double().requires_grad_(True)
    pos = torch.arange(B) * L + ln - 1
    c_ctx = torch.cat([c[pos] for c in cd])
    c_x = xd[pos].repeat(groups, 1)
    hz = c_ctx @ P[0].t()
    h = torch.nn.functional.layer_norm((hz + P[1]) * m_a.double() + c_x, (d,), P[6], P[7], 1e-12)
    z1 = h @ P[2].t()
    a1 = O.act_fn(act)(z1 + P[3])
    z2 = a1 @ P[4].t()
    out = torch.nn.functional.layer_norm((z2 + P[5]) * m_f.double() + h, (d,), P[8], P[9], 1e-12)
    # parameters are trained by the first group's rows only (trainer.py:672-686); inputs receive every row's gradient
    w_in = d_out.double().clone()
    (out * w_in).sum().backward(retain_graph=True)
    d_ctx_ref = [c.grad.clone() for c in cd]
    d_x_ref = None
    # ---- CUDA ----
    dev = 'cuda'
    f = lambda *s: torch.empty(*s, device=dev)        # noqa: E731
    S = dict(ctx=f(C, d), x=f(B, d), hz=f(C, d), st_a=f(C, 2), h=f(C, d), z1=f(C, I), a1=f(C, I), z2=f(C, d), st_f=f(C, 2), out=f(C, d))
    W = [t.to(dev) for t in (Wo, bo, lnAw, lnAb, W1, b1, W2, b2, lnFw, lnFb)]
    cg = [t.to(dev) for t in ctx]
    xg, lng, mag, mfg = x.to(dev), ln.to(dev), m_a.to(dev), m_f.to(dev)
    st = torch.cuda.current_stream().cuda_stream
    aid = A.ops.ACT_IDS[act]
    LIB.call('acsr_tail_fwd', _p(cg[0]), _p(cg[1]) if groups == 2 else None, _p(xg), _p(lng, torch.int64), B, L, d, I, aid,
             _p(W[0]), _p(W[1]), _p(W[2]), _p(W[3]), 1e-12, _p(W[4]), _p(W[5]), _p(W[6]), _p(W[7]), _p(W[8]), _p(W[9]), 1e-12, p,
             _p(mag), _p(mfg), None, 0, 0, _p(S['ctx']), _p(S['x']), _p(S['hz']), _p(S['st_a']), _p(S['h']), _p(S['z1']), _p(S['a1']),
             _p(S['z2']), _p(S['st_f']), _p(S['out']), st)
    close(S['out'], out, 2e-5, 'out')
    close(S['h'], h, 2e-5, 'h')
    close(S['a1'], a1, 2e-5, 'a1')
    close(S['hz'], hz, 1e-5, 'hz')
    assert torch.equal(S['ctx'].cpu(), torch.cat([c[pos] for c in ctx]))
    G = dict(d_z2=f(C, d), d_z1=f(C, I), d_hz=f(C, d), d_x=torch.zeros(groups, T, d, device=dev), d_ctx=torch.zeros(groups, T, d, device=dev))
    gp = [torch.zeros(n, device=dev) for n in (d, d, d, I, d, d, d)]          # bo, lnA_w, lnA_b, b1, b2, lnF_w, lnF_b
    d_out_g = d_out.to(dev)
    LIB.call('acsr_tail_bwd', _p(d_out_g), _p(lng, torch.int64), B, L, d, I, aid, groups, _p(S['x']), _p(S['hz']), _p(S['st_a']),
             _p(S['h']), _p(S['z1']), _p(S['z2']), _p(S['st_f']), _p(W[0]), _p(W[1]), _p(W[2]), _p(W[4]), _p(W[5]), _p(W[6]), _p(W[7]),
             _p(W[8]), p, _p(mag), _p(mfg), None, 0, 0, _p(G['d_z2']), _p(G['d_z1']), _p(G['d_hz']), _p(G['d_x'][0]),
             _p(G['d_x'][1]) if groups == 2 else None, _p(G['d_ctx'][0]), _p(G['d_ctx'][1]) if groups == 2 else None,
             *[_p(t) for t in gp], st)
    for gi in range(groups):
        close(G['d_ctx'][gi], d_ctx_ref[gi], 5e-5, 'd_ctx[%d]' % gi)
    close(G['d_x'].sum(0), xd.grad, 5e-5, 'd_x')
    # parameter gradients: only the first group's rows
    for t in P + cd + [xd]:
        t.grad = None
    w_in[B:] = 0
    (out * w_in).sum().backward()
    for got, ref, name in zip(gp, (P[1], P[6], P[7], P[3], P[5], P[8], P[9]), ('bo', 'lnA_w', 'lnA_b', 'b1', 'b2', 'lnF_w', 'lnF_b')):
        close(got, ref.grad, 1e-4, 'grad ' + name)
    # the weight gradients come from the saved left operands: dW2 = d_z2[:B]^T . a1[:B] etc.
    close(G['d_z2'][:B].double().t() @ S['a1'][:B].double(), P[4].grad, 1e-4, 'dW2')
    close(G['d_z1'][:B].double().t() @ S['h'][:B].double(), P[2].grad, 1e-4, 'dW1')
    close(G['d_hz'][:B].double().t() @ S['ctx'][:B].double(), P[0].grad, 1e-4, 'dWo')


def test_gather_last(A):
    g = torch.Generator().manual_seed(1)
    B, L, d = 9, 50, 64
    xa, xc = torch.randn(B, L, d, generator=g), torch.randn(B, L, d, generator=g)
    ln = torch.randint(1, L + 1, (B,), generator=g)
    ln[0], ln[1] = 1, L
    xac, xcc = xa.clone().cuda().requires_grad_(True), xc.clone().cuda().requires_grad_(True)
    out = A.ops.GatherLastFn.apply(xac, xcc, ln.cuda())
    rows = torch.arange(B)
    assert torch.equal(out[:B].cpu(), xa[rows, ln - 1]) and torch.equal(out[B:].cpu(), xc[rows, ln - 1])
    dy = torch.randn(2 * B, d, generator=g)
    out.backward(dy.cuda())
    ga = torch.zeros_like(xa); ga[rows, ln - 1] = dy[:B]
    gc = torch.zeros_like(xc); gc[rows, ln - 1] = dy[B:]
    assert torch.equal(xac.grad.cpu(), ga) and torch.equal(xcc.grad.cpu(), gc)
    out1 = A.ops.GatherLastFn.apply(None, xcc, ln.cuda())
    assert torch.equal(out1.cpu(), xc[rows, ln - 1])


def test_adam_matches_torch(A):
    g = torch.Generator().manual_seed(2)
    n = 100003
    p0 = torch.randn(n, generator=g)
    pt = p0.clone().requires_grad_(True)
    opt = torch.optim.Adam([pt], lr=1e-3, weight_decay=0.01)
    pc, m, v = p0.clone().cuda(), torch.zeros(n).cuda(), torch.zeros(n).cuda()
    step = torch.zeros(1, dtype=torch.int64).cuda()
    po, mo, vo = p0.clone(), torch.zeros(n), torch.zeros(n)
    for s in range(1, 4):
        gr = torch.randn(n, generator=g)
        pt.grad = gr.clone()
        opt.step()
        A.ops.adam_step(pc, gr.cuda(), m, v, step, 1e-3, weight_decay=0.01)
        po, mo, vo = O.adam_step(po, gr, mo, vo, s, 1e-3, weight_decay=0.01)
    assert int(step.item()) == 3
    close(pc, pt, 1e-6, 'vs torch.optim.Adam')
    close(pc, po, 1e-6, 'vs oracle')


# ----------------------------------------------------------------------------------------------
ATTN_CASES = [
    # H, dh, L, combine, two_level, rich, use_order, use_distance, p
    (2, 32, 50, 'gate', True, 'none', True, True, 0.5),
    (4, 16, 50, 'gate', True, 'none', True, True, 0.5),
    (2, 32, 50, 'gate', True, 'none', True, True, 0.0),
    (8, 16, 50, 'gate', True, 'none', True, True, 0.5),
    (8, 8, 33, 'gate', True, 'none', True, True, 0.3),
    (2, 64, 64, 'gate', True, 'none', True, True, 0.5),
    (2, 32, 20, 'gate', True, 'none', True, True, 0.5),
    (2, 32, 50, 'fixed', True, 'none', True, True, 0.5),
    (2, 32, 50, 'annealing', True, 'none', True, True, 0.5),
    (2, 32, 50, 'gate', False, 'fixed', True, True, 0.5),
    (2, 32, 50, 'fixed', False, 'trainable', True, True, 0.5),
    (2, 32, 50, 'gate', True, 'none', False, True, 0.5),
    (2, 32, 50, 'gate', True, 'none', True, False, 0.5),
    (2, 32, 50, 'gate', True, 'none', False, False, 0.0),
    # sequences longer than 64 (attn_long.cu: key tiles resident, query rows streamed, backward matrices in a workspace);
    # (4, 64, 200) is BASELINE configuration #5's attention shape
    (4, 64, 200, 'gate', True, 'none', True, True, 0.5),
    (2, 32, 80, 'gate', True, 'none', True, True, 0.3),
    (4, 16, 130, 'fixed', False, 'trainable', True, True, 0.5),
    (2, 64, 65, 'annealing', True, 'none', False, True, 0.0),
]
LONG_CASES = [c for c in ATTN_CASES if c[2] > 64]


def _attn_inputs(H, dh, L, combine, two_level, rich, use_order, use_distance, p, seed=0):
    g = torch.Generator().manual_seed(seed + H * 7 + L)
    B, d = 5, H * dh
    cfg = O.default_cfg(n_heads=H, hidden_size=d, combine_option=combine, two_level=two_level,
                        rich_calibrated_combine=rich, use_order=use_order, use_distance=use_distance)
    seq, ln, _ = O.synth_batch(B, L, 50, seed=seed + 1)
    seq[0] = torch.randint(1, 50, (L,), generator=g)          # full row
    t = {k: torch.randn(B, L, d, generator=g) * (1.0 if k in 'mv' else 0.7) for k in ('mq', 'mk', 'mv', 'aq', 'ak')}
    t['gate'] = torch.randn(B, L, L, generator=g) if combine == 'gate' else None
    lp = {}
    if use_order:
        lp['order_affine.weight'] = torch.randn(1, 2 * dh, generator=g) * 0.3
        lp['order_affine.bias'] = torch.randn(1, generator=g) * 0.3
    if use_distance:
        lp['distance_affine.weight'] = torch.randn(1, 2 * dh, generator=g) * 0.3
        lp['distance_affine.bias'] = torch.randn(1, generator=g) * 0.3
        lp['scalar'] = torch.randn(1, generator=g)
    if rich == 'trainable':
        lp['rich_calibrated_combine_ratio'] = torch.tensor([0.35])
    rnd = {}
    if p > 0:
        for k in ('D1', 'D2', 'D3'):
            rnd[(0, k)] = drop((B, H, L, L), p, g)
    rnd[(0, 'noise')] = torch.randn(B, H, L, L, generator=g)
    return cfg, seq, t, lp, rnd, g


def _run_cuda_attn(A, cfg, seq, t, lp, rnd, p, need_att=True, want_probs=True, grad=False, bidirectional=False, plain=False):
    H = cfg['n_heads']
    opts = A.ops.AttnOpts(H, cfg['two_level'], cfg['combine_option'],
                          cfg['rich_calibrated_combine'] if not cfg['two_level'] else 'none', p, bidirectional=bidirectional, plain=plain)
    def c(x):
        if x is None:
            return None
        x = x.clone().cuda()
        return x.requires_grad_(True) if grad else x
    tc = {k: c(v) for k, v in t.items()}
    lpc = {k: c(v) for k, v in lp.items()}
    rand = {k: dev(rnd.get((0, k))) for k in ('D1', 'D2', 'D3', 'noise')}
    out = A.ops.AttnCalibFn.apply(
        tc['mq'], tc['mk'], tc['mv'], tc['aq'], tc['ak'], tc['gate'], seq.cuda(),
        lpc.get('order_affine.weight'), lpc.get('order_affine.bias'), lpc.get('distance_affine.weight'),
        lpc.get('distance_affine.bias'), lpc.get('scalar'), lpc.get('rich_calibrated_combine_ratio'),
        opts, 0.37, p, rand, None, 16, need_att, want_probs)
    return out, tc, lpc


@pytest.mark.parametrize('case', ATTN_CASES)
def test_attn_calib_forward(A, case):
    H, dh, L, combine, two_level, rich, uo, ud, p = case
    cfg, seq, t, lp, rnd, g = _attn_inputs(*case)
    mask = O.additive_mask(seq)
    r = O.attn_calib(t['mq'], t['mk'], t['mv'], t['aq'], t['ak'], t['gate'], mask, lp, cfg, 0, O.Rand(rnd), anneal_rate=0.37)
    (ctx_att, ctx_cal, pen, probs), _, _ = _run_cuda_attn(A, cfg, seq, t, lp, rnd, p)
    names = ['P0', 'P', 'M', 'A', 'C', 'R']
    for i, n in enumerate(names):
        close(probs[i], r[n], 3e-5, n)
    close(ctx_att, r['ctx_att'], 3e-5, 'ctx_att')
    close(ctx_cal, r['ctx_cal'], 3e-5, 'ctx_cal')
    close(pen, r['pen_sq'].view(1), 1e-5, 'pen_sq')
    # masked probabilities are exactly zero (SURVEY a2)
    causal = torch.tril(torch.ones(L, L, dtype=torch.bool))
    assert float(probs[5].cpu()[:, :, ~causal].abs().max()) == 0.0
    # calibrated-only launch gives the same calibrated context
    (na, ctx_cal2, pen2, _), _, _ = _run_cuda_attn(A, cfg, seq, t, lp, rnd, p, need_att=False, want_probs=False)
    assert na is None
    close(ctx_cal2, r['ctx_cal'], 3e-5, 'ctx_cal (cal only)')


@pytest.mark.parametrize('case', ATTN_CASES)
@pytest.mark.parametrize('which', ['both', 'cal', 'att_pen'])
def test_attn_calib_backward(A, case, which):
    H, dh, L, combine, two_level, rich, uo, ud, p = case
    cfg, seq, t, lp, rnd, g = _attn_inputs(*case)
    B, d = t['mq'].shape[0], H * dh
    g_att, g_cal = torch.randn(B, L, d, generator=g), torch.randn(B, L, d, generator=g)
    g_pen = torch.tensor([0.01])
    to = {k: (v.clone().requires_grad_(True) if v is not None else None) for k, v in t.items()}
    lpo = {k: v.clone().requires_grad_(True) for k, v in lp.items()}
    r = O.attn_calib(to['mq'], to['mk'], to['mv'], to['aq'], to['ak'], to['gate'], O.additive_mask(seq), lpo, cfg, 0,
                     O.Rand(rnd), anneal_rate=0.37)
    loss = 0
    if which in ('both', 'cal'):
        loss = loss + (r['ctx_cal'] * g_cal).sum()
    if which in ('both', 'att_pen'):
        loss = loss + (r['ctx_att'] * g_att).sum() + (r['pen_sq'] * g_pen).sum()
    loss.backward()
    (ctx_att, ctx_cal, pen, _), tc, lpc = _run_cuda_attn(A, cfg, seq, t, lp, rnd, p, want_probs=False, grad=True)
    lc = 0
    if which in ('both', 'cal'):
        lc = lc + (ctx_cal * g_cal.cuda()).sum()
    if which in ('both', 'att_pen'):
        lc = lc + (ctx_att * g_att.cuda()).sum() + (pen * g_pen.cuda()).sum()
    lc.backward()
    for k in ('mq', 'mk', 'mv', 'aq', 'ak', 'gate'):
        if to[k] is None:
            continue
        ref = to[k].grad if to[k].grad is not None else torch.zeros_like(to[k])
        got = tc[k].grad if tc[k].grad is not None else torch.zeros_like(tc[k])
        if float(ref.abs().max()) == 0.0:
            assert float(got.abs().max()) < 1e-6, k
        else:
            close(got, ref, 3e-4, 'd_' + k)
    for k in lpo:
        ref = lpo[k].grad if lpo[k].grad is not None else torch.zeros_like(lpo[k])
        got = lpc[k].grad if lpc[k].grad is not None else torch.zeros_like(lpc[k])
        scale = float(ref.abs().max())
        assert float((got.cpu() - ref).abs().max()) <= 5e-4 * scale + 1e-6, (k, got, ref)


def _raw_attn_bwd(A, cfg, seq, t, lp, rnd, p, cots, dual, order=None, ctx_rows=None):
    """raw C-ABI call of the attention backward.  cots = (cal0, pen0, att1, cal1, pen1) device tensors or None."""
    H = cfg['n_heads']
    B, L, d = t['mq'].shape
    dh = d // H
    P = A.ops._p
    c = lambda x: None if x is None else x.clone().cuda().contiguous()
    tc = {k: c(v) for k, v in t.items()}
    lpc = {k: c(v) for k, v in lp.items()}
    rand = {k: c(rnd.get((0, k))) for k in ('D1', 'D2', 'D3', 'noise')}
    seqc = seq.cuda()
    two_level = int(bool(cfg['two_level']))
    comb = A.ops.COMBINE_IDS[cfg['combine_option']]
    rich = A.ops.RICH_IDS.get(cfg['rich_calibrated_combine'], 0) if not cfg['two_level'] else 0
    shared = (P(tc['mq']), P(tc['mk']), P(tc['mv']), P(tc['aq']), P(tc['ak']), P(tc['gate']), P(seqc, torch.int64),
              P(lpc.get('order_affine.weight')), P(lpc.get('order_affine.bias')), P(lpc.get('distance_affine.weight')),
              P(lpc.get('distance_affine.bias')), P(lpc.get('scalar')), B, L, H, dh, two_level, comb, 0.37, rich,
              P(lpc.get('rich_calibrated_combine_ratio')), float(p), P(rand['D1']), P(rand['D2']), P(rand['D3']),
              P(rand['noise']), None, 16)
    S = 2 if dual else 1
    A.ops.attn_workspace(B, L, H, S, torch.device('cuda'))
    out = {k: torch.full((S * B * L, d), float('nan'), device='cuda') for k in ('mq', 'mk', 'mv', 'aq', 'ak')}
    out['gate'] = torch.zeros(S * B * L, L, device='cuda') if tc['gate'] is not None else None
    pg = {k: torch.zeros_like(v) for k, v in lpc.items()}
    outs = (P(out['mq']), P(out['mk']), P(out['mv']), P(out['aq']), P(out['ak']), P(out['gate']),
            P(pg.get('order_affine.weight')), P(pg.get('order_affine.bias')), P(pg.get('distance_affine.weight')),
            P(pg.get('distance_affine.bias')), P(pg.get('scalar')), P(pg.get('rich_calibrated_combine_ratio')))
    cal0, pen0, att1, cal1, pen1 = cots
    st = A.ops._stream()
    if dual:
        A.LIB.call('acsr_attn_calib_bwd2', P(cal0), P(pen0), P(att1), P(cal1), P(pen1), *shared, *outs, P(order, torch.int32), P(ctx_rows, torch.int64), st)
    else:
        A.LIB.call('acsr_attn_calib_bwd', P(att1), P(cal0), P(pen0), *shared, *outs, P(order, torch.int32), P(ctx_rows, torch.int64), st)
    torch.cuda.synchronize()
    return out, pg


@pytest.mark.parametrize('case', [ATTN_CASES[0], ATTN_CASES[1], ATTN_CASES[5], ATTN_CASES[7], ATTN_CASES[9], ATTN_CASES[4]] + LONG_CASES[:3])
@pytest.mark.parametrize('last', [True, False])
def test_attn_calib_backward_two_streams(A, case, last):
    """acsr_attn_calib_bwd2 == two single-stream launches (stream 0: d_cal; stream 1: d_att|d_cal + d_pen);
    cotangent rows that are exactly zero (positions behind len-1) take the skip path."""
    H, dh, L, combine, two_level, rich, uo, ud, p = case
    cfg, seq, t, lp, rnd, g = _attn_inputs(*case)
    B, d = t['mq'].shape[0], H * dh
    g0 = torch.randn(B, L, d, generator=g).cuda()
    g1 = torch.randn(B, L, d, generator=g).cuda()
    g0[1:, 7:] = 0.0                                   # most rows of the calibrated-loss stream carry no cotangent
    if last:
        g1[:, :L - 1] = 0.0
    pen = torch.tensor([0.01]).cuda()
    att1, cal1 = (g1, None) if last else (None, g1)
    order = torch.empty(B, dtype=torch.int32, device='cuda')          # longest-first CTA order must not change results
    A.LIB.call('acsr_seq_order', seq.cuda().data_ptr(), B, L, order.data_ptr(), A.ops._stream())
    nkey = [(int((seq[b] != 0).nonzero().max()) + 1) if bool((seq[b] != 0).any()) else 0 for b in range(B)]
    assert sorted(order.tolist()) == list(range(B)) and all(nkey[order[i]] >= nkey[order[i + 1]] for i in range(B - 1))
    both, pg_both = _raw_attn_bwd(A, cfg, seq, t, lp, rnd, p, (g0, None, att1, cal1, pen), dual=True, order=order)
    s0, pg0 = _raw_attn_bwd(A, cfg, seq, t, lp, rnd, p, (g0, None, None, None, None), dual=False)
    s1, _ = _raw_attn_bwd(A, cfg, seq, t, lp, rnd, p, (cal1, pen, att1, None, None), dual=False)
    T = B * L
    for k in both:
        if both[k] is None:
            continue
        assert not bool(torch.isnan(both[k]).any()), k
        close(both[k][:T], s0[k], 2e-5, 'stream0 d_' + k)
        close(both[k][T:], s1[k], 2e-5, 'stream1 d_' + k)
    for k in pg0:
        scale = float(pg0[k].abs().max())
        assert float((pg_both[k] - pg0[k]).abs().max()) <= 1e-4 * scale + 1e-6, k
    if last:
        # last-layer contract: only context row len-1 carries a cotangent -> the penalty-only row path must give the same
        lens = torch.tensor([int((seq[b] != 0).sum()) for b in range(B)], dtype=torch.int64).cuda()
        h0, h1 = torch.zeros_like(g0), torch.zeros_like(g1)
        ar = torch.arange(B).cuda()
        h0[ar, lens - 1] = g0[ar, lens - 1]
        h1[ar, lens - 1] = g1[ar, lens - 1]
        ref, pg_ref = _raw_attn_bwd(A, cfg, seq, t, lp, rnd, p, (h0, None, h1, None, pen), dual=True)
        got, pg_got = _raw_attn_bwd(A, cfg, seq, t, lp, rnd, p, (h0, None, h1, None, pen), dual=True, order=order, ctx_rows=lens)
        for k in ref:
            if ref[k] is not None:
                close(got[k], ref[k], 2e-5, 'ctx_rows d_' + k)
        for k in pg_ref:
            assert float((pg_got[k] - pg_ref[k]).abs().max()) <= 1e-4 * float(pg_ref[k].abs().max()) + 1e-6, k


def test_attn_long_backward_chunked_workspace(A, monkeypatch):
    """a workspace smaller than the batch: the library walks the batch in chunks of sequences; same gradients."""
    case = LONG_CASES[1]
    H, dh, L, combine, two_level, rich, uo, ud, p = case
    cfg, seq, t, lp, rnd, g = _attn_inputs(*case)
    B, d = t['mq'].shape[0], H * dh
    g0, g1 = torch.randn(B, L, d, generator=g).cuda(), torch.randn(B, L, d, generator=g).cuda()
    pen = torch.tensor([0.01]).cuda()
    ref, pg_ref = _raw_attn_bwd(A, cfg, seq, t, lp, rnd, p, (g0, None, g1, None, pen), dual=True)
    per_seq = A.LIB.query('acsr_attn_workspace_bytes', L, H, 2)
    assert per_seq == ((2 * 2 + 2) * L * L + 2 * 2 * L) * 4 * H
    small = torch.empty(2 * per_seq + 100, dtype=torch.uint8, device='cuda')          # room for 2 of the 5 sequences
    monkeypatch.setattr(A.ops, 'attn_workspace', lambda *a, **k: None)
    try:
        assert A.LIB.query('acsr_set_workspace', small.data_ptr(), small.numel()) == 0
        got, pg_got = _raw_attn_bwd(A, cfg, seq, t, lp, rnd, p, (g0, None, g1, None, pen), dual=True)
        for k in ref:
            if ref[k] is not None:
                close(got[k], ref[k], 1e-5, 'chunked d_' + k)
        for k in pg_ref:
            assert float((pg_got[k] - pg_ref[k]).abs().max()) <= 1e-4 * float(pg_ref[k].abs().max()) + 1e-6, k
        assert A.LIB.query('acsr_set_workspace', small.data_ptr(), per_seq - 4) == 0         # not even one sequence fits
        with pytest.raises(A.AcsrError, match='workspace'):
            _raw_attn_bwd(A, cfg, seq, t, lp, rnd, p, (g0, None, g1, None, pen), dual=True)
    finally:
        ws = A.LIB._ws.get(torch.cuda.current_device())
        A.LIB.query('acsr_set_workspace', ws.data_ptr() if ws is not None else None, ws.numel() if ws is not None else 0)


def test_philox_dropout_and_noise_statistics(A):
    """in-kernel RNG: keep rate, inverted scaling, fwd/bwd reuse the same mask, new step -> new mask."""
    d, T, p = 64, 4096, 0.5
    g = torch.Generator().manual_seed(0)
    h = torch.zeros(T, d).cuda()
    res = torch.zeros(T, d).cuda()
    bias = torch.ones(d).cuda()
    rng = A.ops.DeviceRng(1234, torch.device('cuda'))
    seq = torch.randint(1, 50, (64, 64), generator=g).cuda()
    E = torch.randn(50, d, generator=g).cuda().requires_grad_(True)
    w, b = torch.ones(d).cuda().requires_grad_(True), torch.zeros(d).cuda().requires_grad_(True)
    y1 = A.ops.EmbedLnDropoutFn.apply(seq, E, None, w, b, 1e-12, p, None, rng, 1)
    y_nodrop = A.ops.EmbedLnDropoutFn.apply(seq, E, None, w, b, 1e-12, 0.0, None, None, 1)
    keep = (y1 != 0)
    rate = float(keep.float().mean())
    assert abs(rate - (1 - p)) < 0.01, rate
    close(y1[keep], (y_nodrop / (1 - p))[keep], 1e-6, 'inverted scaling')
    y1b = A.ops.EmbedLnDropoutFn.apply(seq, E, None, w, b, 1e-12, p, None, rng, 1)
    assert torch.equal(y1, y1b)                       # same (seed, step, stream) -> same mask
    y_other_stream = A.ops.EmbedLnDropoutFn.apply(seq, E, None, w, b, 1e-12, p, None, rng, 2)
    assert not torch.equal(y1, y_other_stream)
    # backward regenerates the same mask: compare with the explicit-mask path
    mask = keep.float() / (1 - p)
    dy = torch.randn(y1.shape, generator=g).cuda()
    y1.backward(dy)
    g_philox = E.grad.clone(); E.grad = None
    y2 = A.ops.EmbedLnDropoutFn.apply(seq, E, None, w, b, 1e-12, p, mask, None, 1)
    y2.backward(dy)
    close(g_philox, E.grad, 1e-4, 'bwd mask reuse')     # atomics reorder sums
    rng.advance()
    y3 = A.ops.EmbedLnDropoutFn.apply(seq, E, None, w, b, 1e-12, p, None, rng, 1)
    assert not torch.equal(y1, y3)
    # attention noise ~ N(0,1): A = softmax(noise) when P*M ~ 0 ... check moments through probs_out of M-free setup
    B, H, L, dh = 64, 2, 50, 32
    z = torch.zeros(B, L, H * dh).cuda()
    opts = A.ops.AttnOpts(H, True, 'annealing', 'none', 0.0)
    ids = torch.ones(B, L, dtype=torch.int64).cuda()
    _, _, _, probs = A.ops.AttnCalibFn.apply(z, z, z, z, z, None, ids, None, None, None, None, None, None, opts, 0.5, 0.0,
                                             None, rng, 16, True, True)
    # with zero inputs: P = M = uniform 1/(i+1) on row i; A = softmax(P*M + n(1-M)) ; use last row: M = 1/L
    A_last = probs[3][:, :, L - 1, :]
    n_hat = (torch.log(A_last) - torch.log(A_last).mean(-1, keepdim=True)) / (1 - 1.0 / L)
    assert abs(float(n_hat.std()) - 1.0) < 0.05 and abs(float(n_hat.mean())) < 0.02


# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize('M,V', [(4, 301), (128, 64), (130, 65), (256, 12102), (512, 12102), (300, 1683), (37, 20034)])
def test_logits_store_tcgen05(A, M, V):
    g = torch.Generator().manual_seed(M + V)
    out = torch.randn(M, 64, generator=g)
    E = torch.randn(V, 64, generator=g) * 0.5
    ref = out.double() @ E.double().t()
    s3 = A.ops.logits_scores(out.cuda(), E.cuda(), 3).cpu().double()
    scale = float(ref.abs().max())
    e3 = float((s3 - ref).abs().max()) / scale
    assert e3 < 2e-6, e3                                   # 3xTF32 ~ fp32 sgemm accuracy
    s1 = A.ops.logits_scores(out.cuda(), E.cuda(), 1).cpu().double()
    e1 = float((s1 - ref).abs().max()) / scale
    assert e1 < 1e-3, e1                                   # single-pass TF32 stays inside the 1e-3 budget


@pytest.mark.parametrize('M,V,groups', [(8, 301, 2), (512, 12102, 2), (256, 1683, 1), (6, 65, 2)])
def test_logits_ce_forward_backward(A, M, V, groups):
    g = torch.Generator().manual_seed(M * 3 + V)
    out = torch.randn(M, 64, generator=g) * 2
    E = torch.randn(V, 64, generator=g) * 0.3
    tgt = torch.randint(0, V, (M,), generator=g)
    oo, Eo = out.double().requires_grad_(True), E.double().requires_grad_(True)
    logits = oo @ Eo.t()
    per = M // groups
    ref = torch.stack([torch.nn.functional.cross_entropy(logits[i * per:(i + 1) * per], tgt[i * per:(i + 1) * per])
                       for i in range(groups)])
    wgt = torch.tensor([1.0, -0.7][:groups], dtype=torch.float64)
    (ref * wgt).sum().backward()
    oc, Ec = out.cuda().requires_grad_(True), E.cuda().requires_grad_(True)
    loss = A.ops.LogitsCEFn.apply(oc, Ec, tgt.cuda(), groups, 3)
    close(loss, ref, 1e-5, 'CE loss')                      # north_star: 1e-3
    (loss * wgt.float().cuda()).sum().backward()
    close(oc.grad, oo.grad, 2e-4, 'd_out')
    close(Ec.grad, Eo.grad, 2e-4, 'd_E')


@pytest.mark.parametrize('M,V', [(4, 301), (130, 65), (256, 12102), (512, 12102), (300, 20034), (37, 1000), (1024, 129), (128, 128)])
def test_ce_backward_without_gradient_matrix(A, M, V):
    """acsr_ce_bwd_dout / acsr_ce_bwd_dtable: d_out = G.E and d_E = G^T.out with G = (softmax - onehot) * row_scale recomputed
    inside the kernels (no [M,V] matrix); targets outside [0,V) carry no one-hot (shard-local targets); outputs accumulate."""
    g = torch.Generator().manual_seed(M * 7 + V)
    out = torch.randn(M, 64, generator=g) * 2
    E = torch.randn(V, 64, generator=g) * 0.3
    tgt = torch.randint(-V // 3, V + V // 3, (M,), generator=g)
    tgt[0] = 0
    tgt[-1] = V - 1
    scale = torch.randn(M, generator=g) / M
    scale[M // 2] = 0.0
    logits = out.double() @ E.double().t()
    lse = torch.logsumexp(logits, 1)
    G = torch.exp(logits - lse[:, None])
    ok = (tgt >= 0) & (tgt < V)
    G[torch.nonzero(ok).view(-1), tgt[ok]] -= 1.0
    G = G * scale.double()[:, None]
    base_o = torch.randn(M, 64, generator=g) * 1e-3
    base_e = torch.randn(V, 64, generator=g) * 1e-3
    ref_dout, ref_dE = base_o.double() + G @ E.double(), base_e.double() + G.t() @ out.double()
    oc, Ec, lc, tc, sc = out.cuda(), E.cuda(), lse.float().cuda(), tgt.cuda(), scale.cuda()
    for passes, tol in ((3, 1e-5), (1, 4e-3)):
        d_out = A.ops.ce_bwd_dout(oc, Ec, lc, tc, sc, base_o.cuda(), passes)
        d_E = A.ops.ce_bwd_dtable(oc, Ec, lc, tc, sc, base_e.cuda(), passes)
        close(d_out, ref_dout, tol, 'd_out (passes=%d)' % passes)
        close(d_E, ref_dE, tol, 'd_E (passes=%d)' % passes)
    with pytest.raises(A.AcsrError):
        A.ops.ce_bwd_dout(torch.randn(4, 128).cuda(), torch.randn(9, 128).cuda(), lc[:4], tc[:4], sc[:4], torch.zeros(4, 128).cuda(), 3)


@pytest.mark.parametrize('M,V,k', [(4, 301, 50), (256, 12102, 50), (100, 1683, 50), (7, 70, 10), (130, 20034, 20)])
def test_logits_topk_fused(A, M, V, k):
    g = torch.Generator().manual_seed(M + V + k)
    out = torch.randn(M, 64, generator=g)
    E = torch.randn(V, 64, generator=g) * 0.5
    pos = torch.randint(1, V, (M,), generator=g)
    scores = (out.double() @ E.double().t())
    _, ref_idx = O.full_sort_topk(scores.float(), k)
    for path in ('auto', 'fused', 'fused-private'):   # auto: small catalogues take scores + radix select; fused: streaming top-k (CTAs share a per-row bound) + merge; fused-private: every CTA on its own
        if path == 'auto':
            val, idx, rec = A.ops.full_sort_topk(out.cuda(), E.cuda(), k, pos.cuda(), 3)
        else:
            pv, pi = A.ops.logits_topk_partial(out.cuda(), E.cuda(), k, 0, True, 3, share_bound=(path == 'fused'))
            assert pv.shape[1] == A.ops.logits_num_chunks(M, V)
            val, idx, rec = A.ops.topk_merge(pv, pi, k, pos.cuda())
        idx, val, rec = idx.cpu(), val.cpu(), rec.cpu()
        assert (idx != 0).all() and (idx >= 0).all()            # column 0 is excluded (trainer.py:942)
        assert (val[:, :-1] >= val[:, 1:]).all()                # sorted descending
        close(val, torch.gather(scores, 1, idx), 3e-6, 'top-k scores')
        ok, nbad = O.topk_equal_modulo_ties(idx, ref_idx, scores.float())
        assert ok, nbad
        flags = O.hit_flags(idx, pos)
        assert torch.equal(rec[:, :-1], flags) and (rec[:, -1] == 1).all()


def test_topk_select_ties_and_short_rows(A):
    """exact ties resolve to the lowest item id (stable descending sort); strided rows; k = V - 1."""
    M, V, k = 9, 300, 50
    g = torch.Generator().manual_seed(3)
    sc = torch.randint(0, 12, (M, V + 7), generator=g).float()          # many exact ties, row stride > V
    sc[0] = 1.0                                                          # a constant row
    val, idx, _ = A.ops.topk_select(sc.cuda()[:, :V], k)
    s2 = sc[:, :V].clone()
    s2[:, 0] = -float('inf')
    order = torch.sort(s2, dim=1, descending=True, stable=True)
    assert torch.equal(val.cpu(), order.values[:, :k])
    assert torch.equal(idx.cpu(), order.indices[:, :k])
    val, idx, _ = A.ops.topk_select(sc.cuda()[:, :51], 50)              # k = V - 1: everything but column 0
    assert torch.equal(idx.cpu().sort(dim=1).values, torch.arange(1, 51).expand(M, 50))


# ---- hidden sizes other than 64: scores / CE / CE-gradient on the K-streamed tcgen05 GEMM (gemm_ks.cu epilogues), the streaming
# top-k on the fp32 FMA kernel (logits_simt.cu): same entry points, same contracts ----
@pytest.mark.parametrize('M,V,d', [(4, 301, 128), (130, 65, 256), (256, 12102, 128), (512, 12102, 256), (37, 20034, 32), (300, 1683, 100)])
def test_logits_store_fp32_path(A, M, V, d):
    g = torch.Generator().manual_seed(M + V + d)
    out = torch.randn(M, d, generator=g)
    E = torch.randn(V, d, generator=g) * 0.5
    ref = out.double() @ E.double().t()
    s = A.ops.logits_scores(out.cuda(), E.cuda(), 3).cpu().double()
    e = float((s - ref).abs().max()) / float(ref.abs().max())
    assert e < 4e-6, e          # 3xTF32 on the tensor cores: fp32-level (the K = 256 chain is 96 truncating accumulations)


@pytest.mark.parametrize('M,V,groups,d', [(8, 301, 2, 128), (512, 12102, 2, 256), (256, 1683, 1, 128), (6, 65, 2, 36)])
def test_logits_ce_forward_backward_fp32_path(A, M, V, groups, d):
    g = torch.Generator().manual_seed(M * 3 + V + d)
    out = torch.randn(M, d, generator=g) * (16.0 / d ** 0.5)
    E = torch.randn(V, d, generator=g) * 0.3
    tgt = torch.randint(0, V, (M,), generator=g)
    oo, Eo = out.double().requires_grad_(True), E.double().requires_grad_(True)
    logits = oo @ Eo.t()
    per = M // groups
    ref = torch.stack([torch.nn.functional.cross_entropy(logits[i * per:(i + 1) * per], tgt[i * per:(i + 1) * per])
                       for i in range(groups)])
    wgt = torch.tensor([1.0, -0.7][:groups], dtype=torch.float64)
    (ref * wgt).sum().backward()
    oc, Ec = out.cuda().requires_grad_(True), E.cuda().requires_grad_(True)
    loss = A.ops.LogitsCEFn.apply(oc, Ec, tgt.cuda(), groups, 3)
    close(loss, ref, 1e-5, 'CE loss')
    (loss * wgt.float().cuda()).sum().backward()
    close(oc.grad, oo.grad, 2e-4, 'd_out')
    close(Ec.grad, Eo.grad, 2e-4, 'd_E')


@pytest.mark.parametrize('M,V,k,d', [(4, 301, 50, 128), (256, 12102, 50, 256), (100, 1683, 50, 128), (7, 70, 10, 256), (130, 20034, 20, 128)])
def test_logits_topk_fused_fp32_path(A, M, V, k, d):
    g = torch.Generator().manual_seed(M + V + k + d)
    out = torch.randn(M, d, generator=g)
    E = torch.randn(V, d, generator=g) * 0.5
    pos = torch.randint(1, V, (M,), generator=g)
    scores = (out.double() @ E.double().t())
    _, ref_idx = O.full_sort_topk(scores.float(), k)
    pv, pi = A.ops.logits_topk_partial(out.cuda(), E.cuda(), k, 0, True, 3)
    val, idx, rec = A.ops.topk_merge(pv, pi, k, pos.cuda())
    idx, val, rec = idx.cpu(), val.cpu(), rec.cpu()
    assert (idx != 0).all() and (idx >= 0).all()
    assert (val[:, :-1] >= val[:, 1:]).all()
    close(val, torch.gather(scores, 1, idx), 3e-6, 'top-k scores')
    ok, nbad = O.topk_equal_modulo_ties(idx, ref_idx, scores.float())
    assert ok, nbad
    flags = O.hit_flags(idx, pos)
    assert torch.equal(rec[:, :-1], flags) and (rec[:, -1] == 1).all()


def test_unsupported_shapes_fail_loudly(A):
    with pytest.raises(A.AcsrError):
        A.ops.logits_scores(torch.randn(4, 66).cuda(), torch.randn(10, 66).cuda(), 3)        # d % 4 != 0
    with pytest.raises(A.AcsrError):
        A.ops.logits_scores(torch.randn(4, 64), torch.randn(10, 64), 3)                       # CPU tensors
    with pytest.raises(A.AcsrError):
        A.ops.BiasActFn.apply(torch.randn(4, 6).cuda(), None, 0)                              # n % 4


@pytest.mark.parametrize('T,N,K', [(12800, 64, 64), (12800, 50, 64), (12800, 256, 64), (12800, 64, 256), (777, 128, 128),
                                   (12102, 512, 64), (5, 64, 64), (3000, 1024, 256)])
def test_linear_wgrad_and_linear_fn(A, T, N, K):
    g = torch.Generator().manual_seed(T + N + K)
    dY, X = torch.randn(T, N, generator=g), torch.randn(T, K, generator=g)
    dW, db = A.ops.linear_wgrad(dY.cuda(), X.cuda())
    close(dW, dY.double().t() @ X.double(), 2e-5, 'dW')
    close(db, dY.double().sum(0), 2e-5, 'db')
    # accumulate semantics: a second call adds on top
    dW2, db2 = A.ops.linear_wgrad(dY.cuda(), X.cuda(), dW.clone(), db.clone())
    close(dW2, 2 * (dY.double().t() @ X.double()), 2e-5, 'dW accumulate')
    if T <= 1000:
        W, b = torch.randn(N, K, generator=g), torch.randn(N, generator=g)
        xo, Wo, bo = X.clone().requires_grad_(True), W.clone().requires_grad_(True), b.clone().requires_grad_(True)
        (torch.nn.functional.linear(xo, Wo, bo) * dY).sum().backward()
        xc, Wc, bc = X.clone().cuda().requires_grad_(True), W.clone().cuda().requires_grad_(True), b.clone().cuda().requires_grad_(True)
        y = A.ops.linear(xc.view(1, T, K), Wc, bc)
        assert y.shape == (1, T, N)
        (y * dY.cuda().view(1, T, N)).sum().backward()
        close(xc.grad, xo.grad, 2e-5, 'dx'); close(Wc.grad, Wo.grad, 2e-5, 'dW'); close(bc.grad, bo.grad, 2e-5, 'db')


@pytest.mark.parametrize('rows,N,transposed,bias,acc,batch', [
    (12800, 64, False, True, False, 1), (12800, 256, False, False, False, 1), (12800, 50, False, True, False, 1),
    (25600, 256, True, False, False, 1), (25600, 64, True, False, True, 1), (12800, 64, False, True, False, 3),
    (25600, 64, True, False, True, 2), (77, 64, False, True, False, 1), (1, 130, False, False, True, 1)])
def test_linear_tc(A, rows, N, transposed, bias, acc, batch):
    """tcgen05 linear (3xTF32): Y (+)= X.Wt^T + b against fp64, forward and input-gradient addressing, batched."""
    g = torch.Generator().manual_seed(rows + N + batch)
    X = torch.randn(batch, rows, 64, generator=g)
    W = torch.randn(batch, 64, N, generator=g) * 0.2 if transposed else torch.randn(batch, N, 64, generator=g) * 0.2
    b = torch.randn(batch, N, generator=g) if bias else None
    Y0 = torch.randn(batch, rows, N, generator=g)
    Wt = W.transpose(1, 2) if transposed else W                     # [batch, N, 64]
    ref = X.double() @ Wt.double().transpose(1, 2)
    if bias:
        ref = ref + b.double().unsqueeze(1)
    if acc:
        ref = ref + Y0.double()
    Xc, Wc, Yc = X.cuda(), W.cuda(), Y0.clone().cuda()
    bc = b.cuda() if bias else None
    sn, sk = (1, N) if transposed else (64, 1)
    A.ops.linear_tc(Xc, rows, Wc, N, sn, sk, bc, Yc, N, accumulate=acc, batch=batch, sx=rows * 64, sw=64 * N,
                    sb=N if bias else 0, sy=rows * N)
    close(Yc, ref, 3e-6, 'linear_tc')
    with pytest.raises(A.AcsrError, match='unsupported'):
        A.LIB.call('acsr_linear_tc', Xc.data_ptr(), rows, 128, Wc.data_ptr(), N, 128, 1, None, 0, Yc.data_ptr(), N, 1, 0, 0, 0, 0, 3, None)


# ----------------------------------------------------------------------------------------------
# tcgen05 token-tile GEMMs (acsr_linear_tok*): compared with an fp64 torch reference of the same op
# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize('rows,K,N', [(12800, 64, 64), (300, 64, 256), (1000, 256, 64), (129, 64, 50), (257, 128, 128), (5, 64, 16)])
@pytest.mark.parametrize('accumulate', [False, True])
def test_linear_tok_plain(A, rows, K, N, accumulate):
    g = torch.Generator().manual_seed(rows + K + N)
    X = torch.randn(rows, K, generator=g).cuda()
    W = torch.randn(N, K, generator=g).cuda() * 0.2
    b = torch.randn(N, generator=g).cuda()
    Y0 = torch.randn(rows, N, generator=g).cuda()
    Y = Y0.clone()
    A.ops.linear_tok(X, rows, K, W, N, Y, N, bias=b, accumulate=accumulate)
    ref = X.double() @ W.double().t() + b.double() + (Y0.double() if accumulate else 0)
    close(Y, ref, 3e-6, 'linear_tok')


def test_linear_tok_transposed_kconcat_batched(A):
    g = torch.Generator().manual_seed(5)
    T2, d, I, L = 700, 64, 256, 50
    # input gradient through W2 [d, I]: d_a1 = d_z2 . W2  (weight read transposed)
    dz2 = torch.randn(T2, d, generator=g).cuda()
    W2 = torch.randn(d, I, generator=g).cuda() * 0.1
    da1 = torch.empty(T2, I).cuda()
    A.ops.linear_tok(dz2, T2, d, W2, I, da1, I, w_sn=1, w_sk=I, wkb=64 * I)
    close(da1, dz2.double() @ W2.double(), 3e-6, 'transposed weight')
    # K = 256 with a transposed weight, accumulating: d_h += d_z1 . W1   (W1 [I, d])
    dz1 = torch.randn(T2, I, generator=g).cuda()
    W1 = torch.randn(I, d, generator=g).cuda() * 0.1
    dh0 = torch.randn(T2, d, generator=g).cuda()
    dh = dh0.clone()
    A.ops.linear_tok(dz1, T2, I, W1, d, dh, d, w_sn=1, w_sk=d, wkb=64 * d, accumulate=True)
    close(dh, dh0.double() + dz1.double() @ W1.double(), 3e-6, 'K=256 accumulate')
    # K-concatenated stacked operands: d_x += sum_b d_qkv[b] . Wqkv[b]
    dqkv = torch.randn(3, T2, d, generator=g).cuda()
    Wqkv = torch.randn(3, d, d, generator=g).cuda() * 0.1
    dx0 = torch.randn(T2, d, generator=g).cuda()
    dx = dx0.clone()
    A.ops.linear_tok(dqkv, T2, 3 * d, Wqkv, d, dx, d, ldx=d, xkb=T2 * d, w_sn=1, w_sk=d, wkb=d * d, accumulate=True)
    ref = dx0.double() + sum(dqkv[i].double() @ Wqkv[i].double() for i in range(3))
    close(dx, ref, 3e-6, 'K-concat')
    # rows of a leading sub-range only
    dx2 = dx0.clone()
    A.ops.linear_tok(dqkv, 300, 3 * d, Wqkv, d, dx2, d, ldx=d, xkb=T2 * d, w_sn=1, w_sk=d, wkb=d * d, accumulate=True)
    close(dx2[:300], ref[:300], 3e-6, 'K-concat rows')
    assert torch.equal(dx2[300:], dx0[300:])
    # batched with a shared input: Q/K/V projections
    x = torch.randn(T2, d, generator=g).cuda()
    bq = torch.randn(3, d, generator=g).cuda()
    qkv = torch.empty(3, T2, d).cuda()
    A.ops.linear_tok(x, T2, d, Wqkv, d, qkv, d, bias=bq, batch=3, sx=0, sw=d * d, sb=d, sy=T2 * d)
    for i in range(3):
        close(qkv[i], x.double() @ Wqkv[i].double().t() + bq[i].double(), 3e-6, 'batched %d' % i)
    # unaligned rows (gate: K = L = 50 input gradient, N = 50 forward)
    Wg = torch.randn(L, d, generator=g).cuda() * 0.1
    bg = torch.randn(L, generator=g).cuda()
    gl = torch.empty(T2, L).cuda()
    A.ops.linear_tok(x, T2, d, Wg, L, gl, L, bias=bg)
    close(gl, x.double() @ Wg.double().t() + bg.double(), 3e-6, 'N=50')
    dgl = torch.randn(T2, L, generator=g).cuda()
    dmq0 = torch.randn(T2, d, generator=g).cuda()
    dmq = dmq0.clone()
    A.ops.linear_tok(dgl, T2, L, Wg, d, dmq, d, ldx=L, w_sn=1, w_sk=d, wkb=64 * d, accumulate=True)
    close(dmq, dmq0.double() + dgl.double() @ Wg.double(), 3e-6, 'K=50')


@pytest.mark.parametrize('K,p,explicit', [(64, 0.0, False), (64, 0.5, True), (256, 0.5, True), (64, 0.5, False), (128, 0.3, True)])
def test_linear_tok_bdrl(A, K, p, explicit):
    g = torch.Generator().manual_seed(K + int(p * 10))
    R, Tres, d = 2 * 640, 640, 64
    X = torch.randn(R, K, generator=g).cuda()
    W = torch.randn(d, K, generator=g).cuda() * 0.2
    b = torch.randn(d, generator=g).cuda()
    res = torch.randn(Tres, d, generator=g).cuda()
    lw, lb = torch.randn(d, generator=g).cuda(), torch.randn(d, generator=g).cuda()
    mask = drop((R, d), p, g).cuda() if explicit else None
    rng = A.ops.DeviceRng(77, torch.device('cuda'))
    HZ, out, stats = torch.empty(R, d).cuda(), torch.empty(R, d).cuda(), torch.empty(R, 2).cuda()
    A.ops.linear_tok_bdrl(X, R, K, W, b, res, Tres, lw, lb, 1e-12, p, mask, rng.ptr, 19, HZ, out, stats)
    hz = X.double() @ W.double().t()
    close(HZ, hz, 3e-6, 'HZ')
    # the unfused kernel with the same rng / mask is the reference of the epilogue (same Philox counters)
    out2, stats2 = torch.empty(R, d).cuda(), torch.empty(R, 2).cuda()
    A.LIB.call('acsr_bias_dropout_res_ln_fwd', HZ.data_ptr(), b.data_ptr(), res.data_ptr(), lw.data_ptr(), lb.data_ptr(), 1e-12,
               R, d, Tres, p, mask.data_ptr() if explicit else None, rng.ptr, 19, out2.data_ptr(), stats2.data_ptr(),
               A.ops._stream())
    close(out, out2, 2e-5, 'out vs unfused')
    close(stats, stats2, 2e-5, 'stats vs unfused')
    if explicit or p == 0.0:
        m = mask.double() if explicit else 1.0
        x = (hz + b.double()) * m + res.double().repeat(R // Tres, 1)
        mean = x.mean(-1, keepdim=True)
        var = ((x - mean) ** 2).mean(-1, keepdim=True)
        ref = (x - mean) / torch.sqrt(var + 1e-12) * lw.double() + lb.double()
        close(out, ref, 2e-5, 'out')


def test_ce_finalize_losses_equals_separate_kernels(A):
    """single-launch CE finalize + adversarial-loss glue == acsr_ce_finalize followed by acsr_loss_combine."""
    M, V, d, N = 512, 3001, 64, 3
    g = torch.Generator().manual_seed(5)
    out, E = torch.randn(M, d, generator=g).cuda(), (torch.randn(V, d, generator=g) * 0.3).cuda()
    tgt = torch.randint(0, V, (M,), generator=g).cuda()
    pen = (torch.rand(N, generator=g).double() * 1000 + 10).cuda()
    part = A.ops.ce_partial(out, E, 3)
    lse, tl, rl, loss = A.ops.ce_finalize(part, out, E, tgt, 2)
    P = A.ops._p
    la, dp = torch.empty(1, device='cuda'), torch.empty(N, device='cuda')
    A.LIB.call('acsr_loss_combine', pen.data_ptr(), N, P(loss[1:]), None, 0.03, P(la), P(dp), A.ops._stream())
    lse2, tl2, rl2, loss2 = (torch.empty_like(t) for t in (lse, tl, rl, loss))
    la2, dp2 = torch.empty_like(la), torch.empty_like(dp)
    cnt = torch.zeros(1, dtype=torch.int32, device='cuda')
    A.LIB.call('acsr_ce_finalize_losses', P(part), part.shape[1], P(out), P(E), P(tgt, torch.int64), M, d, V, 0, 2, P(lse2), P(tl2),
               P(rl2), P(loss2), pen.data_ptr(), N, None, 0.03, P(la2), P(dp2), cnt.data_ptr(), A.ops._stream())
    assert int(cnt.item()) == 0                           # the last CTA resets the arrival counter
    for a, b in ((lse, lse2), (tl, tl2), (rl, rl2), (loss, loss2), (la, la2), (dp, dp2)):
        assert torch.equal(a, b)
    ref = torch.nn.functional.cross_entropy((out.double() @ E.double().t())[:M // 2], tgt[:M // 2])
    assert abs(float(loss2[0]) - float(ref)) < 1e-5 * abs(float(ref))


def test_attention_edge_rows(A):
    """edge inputs the reference handles: a batch of one, a sequence of one item, a full-length row, L = 1."""
    for (B, L, H, dh) in ((1, 50, 2, 32), (3, 1, 2, 32), (2, 7, 1, 16)):
        case = (H, dh, L, 'gate', True, 'none', True, True, 0.0)
        cfg, seq, t, lp, rnd, g = _attn_inputs(*case)
        seq, t = seq[:B].clone(), {k: (v[:B].clone() if v is not None else None) for k, v in t.items()}
        rnd = {k: v[:B].clone() for k, v in rnd.items()}
        seq[0] = torch.randint(1, 50, (L,), generator=g)
        if B > 1:
            seq[1] = 0
            seq[1, 0] = 7                                   # a single item followed by padding
        r = O.attn_calib(t['mq'], t['mk'], t['mv'], t['aq'], t['ak'], t['gate'], O.additive_mask(seq), lp, cfg, 0, O.Rand(rnd), anneal_rate=0.37)
        (ctx_att, ctx_cal, pen, probs), _, _ = _run_cuda_attn(A, cfg, seq, t, lp, rnd, 0.0)
        close(ctx_att, r['ctx_att'], 3e-5, 'ctx_att')
        close(ctx_cal, r['ctx_cal'], 3e-5, 'ctx_cal')
        close(pen, r['pen_sq'].view(1), 1e-5, 'pen_sq')


def test_fold_attack_weights(A):
    """{Wq, Wk, Wv, Waq.Wq, Wak.Wk} and the matching biases: attack_q = x.(Waq.Wq)^T + (Waq.bq + baq)."""
    d = 64
    g = torch.Generator().manual_seed(9)
    Wqkv, bqkv = torch.randn(3, d, d, generator=g) * 0.1, torch.randn(3, d, generator=g) * 0.1
    Waqk, baqk = torch.randn(2, d, d, generator=g) * 0.1, torch.randn(2, d, generator=g) * 0.1
    oW, ob = torch.empty(5, d, d, device='cuda'), torch.empty(5, d, device='cuda')
    P = A.ops._p
    dev = [t.cuda() for t in (Wqkv, bqkv, Waqk, baqk)]                  # keep the device copies alive across the launch
    A.LIB.call('acsr_fold_attack_weights', P(dev[0]), P(dev[1]), P(dev[2]), P(dev[3]), d, P(oW), P(ob), A.ops._stream())
    torch.cuda.synchronize()
    assert torch.equal(oW[:3].cpu(), Wqkv) and torch.equal(ob[:3].cpu(), bqkv)
    x = torch.randn(7, d, generator=g).double()
    for i in range(2):
        ref = (x @ Wqkv[i].double().t() + bqkv[i].double()) @ Waqk[i].double().t() + baqk[i].double()
        got = x @ oW[3 + i].cpu().double().t() + ob[3 + i].cpu().double()
        close(got, ref, 2e-5, 'folded attack projection %d' % i)



# bidirectional attention mask (AcBERT4Rec: get_attention_mask(item_seq, bidirectional=True), abstract_recommender.py:136-143)
BIDIR_CASES = [ATTN_CASES[i] for i in (0, 1, 4, 5, 7, 9, 10, 13)] + [(2, 32, 51, 'fixed', True, 'none', True, True, 0.5)]


@pytest.mark.parametrize('case', BIDIR_CASES)
def test_attn_calib_bidirectional_forward_backward(A, case):
    """only padded keys are masked: rows see keys j > i (both branches of the order calibrator in play); forward
    probabilities / contexts / penalty and every gradient against the oracle with the bidirectional additive mask."""
    H, dh, L, combine, two_level, rich, uo, ud, p = case
    cfg, seq, t, lp, rnd, g = _attn_inputs(*case)
    B, d = t['mq'].shape[0], H * dh
    mask = O.additive_mask(seq, bidirectional=True)
    g_att, g_cal = torch.randn(B, L, d, generator=g), torch.randn(B, L, d, generator=g)
    g_pen = torch.tensor([0.01])
    to = {k: (v.clone().requires_grad_(True) if v is not None else None) for k, v in t.items()}
    lpo = {k: v.clone().requires_grad_(True) for k, v in lp.items()}
    r = O.attn_calib(to['mq'], to['mk'], to['mv'], to['aq'], to['ak'], to['gate'], mask, lpo, cfg, 0, O.Rand(rnd), anneal_rate=0.37)
    ((r['ctx_cal'] * g_cal).sum() + (r['ctx_att'] * g_att).sum() + (r['pen_sq'] * g_pen).sum()).backward()
    (ctx_att, ctx_cal, pen, probs), _, _ = _run_cuda_attn(A, cfg, seq, t, lp, rnd, p, bidirectional=True)
    for i, n in enumerate(['P0', 'P', 'M', 'A', 'C', 'R']):
        close(probs[i], r[n].detach(), 3e-5, n)
    close(ctx_att, r['ctx_att'].detach(), 3e-5, 'ctx_att')
    close(ctx_cal, r['ctx_cal'].detach(), 3e-5, 'ctx_cal')
    close(pen, r['pen_sq'].detach().view(1), 1e-5, 'pen_sq')
    # rows really see later keys: the upper triangle of a full-length row carries probability mass
    upper = torch.triu(torch.ones(L, L, dtype=torch.bool), 1)
    assert float(probs[5].cpu()[0][:, upper].abs().max()) > 0.0
    (ctx_att, ctx_cal, pen, _), tc, lpc = _run_cuda_attn(A, cfg, seq, t, lp, rnd, p, want_probs=False, grad=True, bidirectional=True)
    ((ctx_cal * g_cal.cuda()).sum() + (ctx_att * g_att.cuda()).sum() + (pen * g_pen.cuda()).sum()).backward()
    for k in ('mq', 'mk', 'mv', 'aq', 'ak', 'gate'):
        if to[k] is None:
            continue
        close(tc[k].grad, to[k].grad, 3e-4, 'd_' + k)
    for k in lpo:
        ref = lpo[k].grad if lpo[k].grad is not None else torch.zeros_like(lpo[k])
        got = lpc[k].grad if lpc[k].grad is not None else torch.zeros_like(lpc[k])
        scale = float(ref.abs().max())
        assert float((got.cpu() - ref).abs().max()) <= 5e-4 * scale + 1e-6, (k, got, ref)


# the layer of transformer_layers.py:873-953 (ACSSEPT): attacked / calibrated / combined attention WITHOUT the re-normalising softmaxes
PLAIN_CASES = [ATTN_CASES[i] for i in (0, 1, 4, 5, 7, 9, 10, 13)] + [(2, 32, 50, 'gate', True, 'none', True, True, 0.5),
                                                                     (4, 32, 50, 'fixed', False, 'trainable', True, True, 0.5)]
PLAIN_CASES = [c for c in PLAIN_CASES if c[2] <= 64]


@pytest.mark.parametrize('case', PLAIN_CASES)
def test_attn_calib_transformer_layers_variant(A, case):
    """ACSR_ATTN_PLAIN: A = origin*M + noise*(1-M), C = origin*exp(1-M) and the combination are used as computed
    (transformer_layers.py:919-927).  Masked keys keep the bare noise as attacked weight, so every key of a row is in play;
    forward probabilities / contexts / penalty and every gradient against the oracle restatement of that variant."""
    H, dh, L, combine, two_level, rich, uo, ud, p = case
    cfg, seq, t, lp, rnd, g = _attn_inputs(*case)
    cfg['attn_variant'] = 'transformer_layers'
    B, d = t['mq'].shape[0], H * dh
    mask = O.additive_mask(seq)
    g_att, g_cal = torch.randn(B, L, d, generator=g), torch.randn(B, L, d, generator=g)
    g_pen = torch.tensor([0.01])
    to = {k: (v.clone().requires_grad_(True) if v is not None else None) for k, v in t.items()}
    lpo = {k: v.clone().requires_grad_(True) for k, v in lp.items()}
    r = O.attn_calib(to['mq'], to['mk'], to['mv'], to['aq'], to['ak'], to['gate'], mask, lpo, cfg, 0, O.Rand(rnd), anneal_rate=0.37)
    ((r['ctx_cal'] * g_cal).sum() + (r['ctx_att'] * g_att).sum() + (r['pen_sq'] * g_pen).sum()).backward()
    (ctx_att, ctx_cal, pen, probs), _, _ = _run_cuda_attn(A, cfg, seq, t, lp, rnd, p, plain=True)
    for i, n in enumerate(['P0', 'P', 'M', 'A', 'C', 'R']):
        close(probs[i], r[n].detach(), 3e-5, n)
    close(ctx_att, r['ctx_att'].detach(), 3e-5, 'ctx_att')
    close(ctx_cal, r['ctx_cal'].detach(), 3e-5, 'ctx_cal')
    close(pen, r['pen_sq'].detach().view(1), 1e-5, 'pen_sq')
    # the attacked weights of future keys are the noise itself
    upper = torch.triu(torch.ones(L, L, dtype=torch.bool), 1)
    assert torch.equal(probs[3].cpu()[0][:, upper], rnd[(0, 'noise')][0][:, upper])
    (ctx_att, ctx_cal, pen, _), tc, lpc = _run_cuda_attn(A, cfg, seq, t, lp, rnd, p, want_probs=False, grad=True, plain=True)
    ((ctx_cal * g_cal.cuda()).sum() + (ctx_att * g_att.cuda()).sum() + (pen * g_pen.cuda()).sum()).backward()
    for k in ('mq', 'mk', 'mv', 'aq', 'ak', 'gate'):
        if to[k] is None:
            continue
        close(tc[k].grad, to[k].grad, 3e-4, 'd_' + k)
    for k in lpo:
        ref = lpo[k].grad if lpo[k].grad is not None else torch.zeros_like(lpo[k])
        got = lpc[k].grad if lpc[k].grad is not None else torch.zeros_like(lpc[k])
        scale = float(ref.abs().max())
        assert float((got.cpu() - ref).abs().max()) <= 5e-4 * scale + 1e-6, (k, got, ref)
    # calibrated stream alone (evaluation, non-final layers): no attacked context asked for
    (na, ctx_cal2, pen2, _), _, _ = _run_cuda_attn(A, cfg, seq, t, lp, rnd, p, need_att=False, want_probs=False, plain=True)
    assert na is None
    close(ctx_cal2, r['ctx_cal'].detach(), 3e-5, 'ctx_cal (calibrated only)')


# ---- ACTiSASRec: time-interval aware terms (timeaware.cu) ----
def _pair_ref(P, T, tmat, Dp, Dt):
    """E[b,i,j,c] = P[j,c]*Dp[b,j,c] + T[t[b,i,j],c]*Dt[b,i,j,c] in double"""
    return (P.double().unsqueeze(0) * Dp.double()).unsqueeze(1) + T.double()[tmat.long()] * Dt.double()


@pytest.mark.parametrize('shape', [(3, 50, 2, 32, 17, 0.5), (2, 23, 4, 8, 256, 0.0), (5, 64, 1, 64, 40, 0.3), (2, 50, 2, 128, 256, 0.5)])
def test_time_aware_pair_kernels(A, shape):
    """pair_score / pair_context / pair_wgrad and the interval matrix against a dense double-precision restatement of
    actisasrec.py:110-124, 146-155 and transformer_layers.py:1085-1091, 1128-1134 (explicit dropout multipliers)"""
    B, L, H, dh, span, p = shape
    d = H * dh
    g = torch.Generator().manual_seed(B * 100 + L)
    ts = (torch.cumsum(torch.randint(0, 2 * max(span // L, 2), (B, L), generator=g), 1) + 1000).float()
    ts[1, L // 2:] = 0.0                                         # a padded tail
    tmat = A.ops.time_matrix(ts.cuda(), span)
    want_t = (ts.unsqueeze(-1) - ts.unsqueeze(1)).abs().clamp(max=span).int()
    assert torch.equal(tmat.cpu(), want_t) and tmat.dtype == torch.int32
    P, T = torch.randn(L, d, generator=g) * 0.5, torch.randn(span + 1, d, generator=g) * 0.5
    Dp = drop((B, L, d), p, g) if p > 0 else torch.ones(B, L, d)
    Dt = drop((B, L, L, d), p, g) if p > 0 else torch.ones(B, L, L, d)
    x = torch.randn(B, L, d, generator=g)
    prob = torch.randn(B, H, L, L, generator=g)
    gs, gy = torch.randn(B, H, L, L, generator=g), torch.randn(B, L, d, generator=g)
    # reference in double
    Pd, Td, xd, pd = (t.clone().double().requires_grad_(True) for t in (P, T, x, prob))
    E = (Pd.unsqueeze(0) * Dp.double()).unsqueeze(1) + torch.nn.functional.embedding(want_t.long(), Td, padding_idx=0) * Dt.double()
    Eh = E.view(B, L, L, H, dh).permute(0, 3, 1, 2, 4)           # [B,H,L,L,dh]
    s_ref = (Eh @ xd.view(B, L, H, dh).permute(0, 2, 1, 3).unsqueeze(-1)).squeeze(-1)
    y_ref = (pd.unsqueeze(-2) @ Eh).squeeze(-2).permute(0, 2, 1, 3).reshape(B, L, d)
    causal = torch.tril(torch.ones(L, L)).bool()
    ((s_ref * gs.double() * causal).sum() + (y_ref * gy.double()).sum()).backward()
    spec = A.ops.PairSpec(tmat, H, p, Dp.cuda() if p > 0 else None, Dt.cuda() if p > 0 else None)
    Pc, Tc, xc, pc = (t.clone().cuda().requires_grad_(True) for t in (P, T, x, prob))
    s = A.ops.PairScoreFn.apply(xc, Pc, Tc, spec, 1)
    y = A.ops.PairContextFn.apply(pc, Pc, Tc, spec)
    close(s, (s_ref * causal).detach(), 2e-5, 'pair score')
    assert float(s.cpu()[:, :, ~causal].abs().max()) == 0.0
    close(y, y_ref.detach(), 2e-5, 'pair context')
    ((s * gs.cuda()).sum() + (y * gy.cuda()).sum()).backward()
    close(xc.grad, xd.grad, 3e-5, 'd x')
    close(pc.grad, pd.grad, 3e-5, 'd prob')
    want_dP = Pd.grad.clone()
    want_dP[0] = 0                                               # nn.Embedding(padding_idx=0) on the position ids (actisasrec.py:55-56)
    close(Pc.grad, want_dP, 5e-5, 'd position table')
    close(Tc.grad, Td.grad, 5e-5, 'd interval table')
    assert float(Tc.grad[0].abs().max()) == 0.0


def test_time_aware_philox_dropout_is_consistent(A):
    """with Philox multipliers forward and backward must draw the same masks: the kernels are linear in x / prob, so the
    gradient against a fixed cotangent equals the finite response of the forward"""
    B, L, H, dh, span, p = 2, 50, 2, 32, 30, 0.5
    d = H * dh
    g = torch.Generator().manual_seed(5)
    ts = (torch.cumsum(torch.randint(0, 5, (B, L), generator=g), 1) + 10).float().cuda()
    tmat = A.ops.time_matrix(ts, span)
    rng = A.ops.DeviceRng(123, torch.device('cuda'))
    rng.advance()
    spec = A.ops.PairSpec(tmat, H, p, None, None, rng, 2, 4)
    P, T = (torch.randn(L, d, generator=g) * 0.5).cuda(), (torch.randn(span + 1, d, generator=g) * 0.5).cuda()
    x = torch.randn(B, L, d, generator=g).cuda().requires_grad_(True)
    gs = torch.randn(B, H, L, L, generator=g).cuda()
    s1 = A.ops.PairScoreFn.apply(x, P, T, spec, 0)
    s2 = A.ops.PairScoreFn.apply(x, P, T, spec, 0)
    assert torch.equal(s1, s2)
    keep = float((A.ops.PairScoreFn.apply(torch.ones_like(x), torch.zeros_like(P), torch.ones_like(T), spec, 0)).mean()) / dh
    assert abs(keep - 1.0) < 0.05                               # E[multiplier] == 1 (inverted dropout)
    (s1 * gs).sum().backward()
    x2 = torch.randn(B, L, d, generator=g).cuda()
    lhs = float((A.ops.PairScoreFn.apply(x2, P, T, spec, 0) * gs).sum())
    rhs = float((x.grad * x2).sum())
    assert abs(lhs - rhs) <= 2e-4 * max(abs(lhs), 1.0)


def test_gather_rows_and_weighted_ce(A):
    """the two pieces AcBERT4Rec adds around the encoder (acbert4rec.py:198-222): row gather (+ scatter-add backward) and the
    masked-item cross entropy with per-row weights."""
    g = torch.Generator().manual_seed(3)
    T, d, n, V = 300, 64, 77, 501
    x = torch.randn(T, d, generator=g)
    idx = torch.randint(0, T, (n,), generator=g)
    idx[0] = 0
    xc = x.clone().cuda().requires_grad_(True)
    y = A.ops.GatherRowsFn.apply(xc, idx.cuda())
    assert torch.equal(y.detach().cpu(), x[idx])
    gy = torch.randn(n, d, generator=g)
    y.backward(gy.cuda())
    want = torch.zeros(T, d).index_add_(0, idx, gy)
    close(xc.grad, want, 1e-6, 'gather backward')
    out = (torch.randn(2 * n, d, generator=g) * 0.7)
    E = (torch.randn(V, d, generator=g) * 0.3)
    tgt = torch.randint(0, V, (2 * n,), generator=g)
    w = (torch.rand(2 * n, generator=g) > 0.4).float()
    oo, Eo = out.clone().double().requires_grad_(True), E.clone().double().requires_grad_(True)
    lg = oo @ Eo.t()
    rl = torch.logsumexp(lg, 1) - lg[torch.arange(2 * n), tgt]
    want_loss = torch.stack([(rl[:n] * w[:n].double()).sum() / w[:n].sum(), (rl[n:] * w[n:].double()).sum() / w[n:].sum()])
    (want_loss[0] * 0.7 - want_loss[1] * 1.3).backward()
    oc, Ec = out.clone().cuda().requires_grad_(True), E.clone().cuda().requires_grad_(True)
    loss = A.ops.LogitsCEFn.apply(oc, Ec, tgt.cuda(), 2, 3, w.cuda())
    close(loss, want_loss, 1e-5, 'weighted CE')
    (loss[0] * 0.7 - loss[1] * 1.3).backward()
    close(oc.grad, oo.grad, 2e-4, 'd_out')
    close(Ec.grad, Eo.grad, 2e-4, 'd_table')
