"""acsr_dense_bwd: the backward of a layer's dense part after its attention in one launch, against a float64 restatement of the
chain it replaces (FFN LayerNorm backward, d_a1 = d_z2.W2, activation backward, d_h += d_z1.W1, attention LayerNorm backward,
d_ctx = d_hz.Wo) and against that chain run as its six launches.  Dropout masks: explicit, Philox (the counters of the forward's
acsr_linear_tok_bdrl), and p = 0.  Tolerances: 1e-4 of the tensor's max |value| with 3xTF32 (DESIGN.md section 2 allows 1e-3),
5e-3 with one TF32 product."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

D = 64
EPS = 1e-12
P_DROP = 0.5
STREAM_A, STREAM_F = 19, 21


@pytest.fixture(scope='module')
def A():
    import ac_tsr_b200 as pkg
    pkg.LIB.load()
    return pkg


def close(a, b, rtol, what=''):
    a = a.detach().double()
    b = b.detach().double()
    scale = float(b.abs().max().clamp(min=1e-30))
    err = float((a - b).abs().max())
    assert err <= rtol * scale + 1e-12, '%s: err %.3e scale %.3e' % (what, err, scale)


def philox_masks(A, rng, stream, rows):
    """the multipliers acsr_linear_tok_bdrl's forward draws for rows [0, rows): its LayerNorm of (0.X^T + 1) * m + 0 with unit
    weight is (m - mean) * rstd, which gives m back exactly (m is 0 or 1 / (1 - p))"""
    z = torch.zeros(rows, D, device='cuda')
    hz, out, st = torch.empty_like(z), torch.empty_like(z), torch.empty(rows, 2, device='cuda')
    A.ops.linear_tok_bdrl(z, rows, D, torch.zeros(D, D, device='cuda'), torch.ones(D, device='cuda'), z, rows,
                          torch.ones(D, device='cuda'), torch.zeros(D, device='cuda'), EPS, P_DROP, None, rng.ptr, stream, hz, out, st)
    m = out.double() / st[:, 1:].double() + st[:, :1].double()
    keep = 1.0 / (1.0 - P_DROP)
    return torch.where(m > 0.5 * keep, torch.full_like(m, keep), torch.zeros_like(m)).float()


def make(A, rows, act_rows, res_rows, I, seed, mode):
    """inputs of one call; mode 'mask' (explicit masks), 'philox' (device RNG) or 'none' (p = 0).  The saved statistics are those
    of the forward on the saved tensors.  -> (tensors, masks as float64 [act_rows, 64] for the reference)"""
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g)             # noqa: E731
    t = dict(d_out=r(rows, D), z2=r(act_rows, D), h=r(act_rows, D), z1=r(act_rows, I), hz=r(act_rows, D), x_res=r(res_rows, D),
             b2=r(D) * 0.1, bo=r(D) * 0.1, b1=r(I) * 0.1, lnF_w=1 + 0.2 * r(D), lnA_w=1 + 0.2 * r(D),
             W2=r(D, I) * 0.1, W1=r(I, D) * 0.1, Wo=r(D, D) * 0.1)
    t = {k: v.cuda() for k, v in t.items()}
    t['rng'] = None
    if mode == 'mask':
        keep = torch.rand(2, act_rows, D, generator=g) > P_DROP
        m = (keep.float() / (1 - P_DROP)).cuda()
        t['m_f'], t['m_a'] = m[0].contiguous(), m[1].contiguous()
        masks = (t['m_f'], t['m_a'])
    elif mode == 'philox':
        t['m_f'] = t['m_a'] = None
        t['rng'] = A.ops.DeviceRng(seed, torch.device('cuda'))
        masks = (philox_masks(A, t['rng'], STREAM_F, act_rows), philox_masks(A, t['rng'], STREAM_A, act_rows))
    else:
        t['m_f'] = t['m_a'] = None
        one = torch.ones(act_rows, D, device='cuda')
        masks = (one, one)
    t['p'] = 0.0 if mode == 'none' else P_DROP
    ridx = torch.arange(act_rows, device='cuda') % res_rows
    for pre, st, m in (((t['z2'] + t['b2']) * masks[0] + t['h'], 'st_f', masks[0]),
                       ((t['hz'] + t['bo']) * masks[1] + t['x_res'][ridx], 'st_a', masks[1])):
        mean, var = pre.mean(1), pre.var(1, unbiased=False)
        t[st] = torch.stack((mean, 1.0 / torch.sqrt(var + EPS)), 1).contiguous()
    return t, [x.double() for x in masks]


def act_grad(act, x):
    if act == 0:
        return 0.5 * (1 + torch.erf(x / math.sqrt(2))) + x * torch.exp(-0.5 * x * x) / math.sqrt(2 * math.pi)
    if act == 1:
        return (x > 0).double()
    s = torch.sigmoid(x)
    if act == 2:
        return s + x * s * (1 - s)
    if act == 3:
        return 1 - torch.tanh(x) ** 2
    return s * (1 - s)


def reference(t, masks, rows, act_rows, res_rows, param_rows, act):
    """float64 restatement of the six-launch chain -> dict of the kernel's outputs (LayerNorm gradients as increments)"""
    q = {k: (v.double() if torch.is_tensor(v) else v) for k, v in t.items()}
    ia = torch.arange(rows, device='cuda') % act_rows
    ir = torch.arange(rows, device='cuda') % res_rows

    def ln_bwd(g, pre, bias, res, w, st, m):
        xh = ((pre + bias) * m + res - st[:, :1]) * st[:, 1:]
        gw = g * w
        d_res = st[:, 1:] * (gw - gw.mean(1, keepdim=True) - xh * (gw * xh).mean(1, keepdim=True))
        return d_res, d_res * m, (g * xh)[:param_rows].sum(0), g[:param_rows].sum(0)

    d_pre, d_z2, gFw, gFb = ln_bwd(q['d_out'], q['z2'][ia], q['b2'], q['h'][ia], q['lnF_w'], q['st_f'][ia], masks[0][ia])
    d_z1 = (d_z2 @ q['W2']) * act_grad(act, q['z1'][ia] + q['b1'])
    d_h = d_pre + d_z1 @ q['W1']
    d_xres, d_hz, gAw, gAb = ln_bwd(d_h, q['hz'][ia], q['bo'], q['x_res'][ir], q['lnA_w'], q['st_a'][ia], masks[1][ia])
    return dict(d_z2=d_z2, d_z1=d_z1, d_hz=d_hz, d_xres=d_xres, d_ctx=d_hz @ q['Wo'], gFw=gFw, gFb=gFb, gAw=gAw, gAb=gAb)


def outputs(t, rows, I, seed):
    """output buffers pre-filled with nonzero values: overwritten rows and untouched rows both show"""
    g = torch.Generator().manual_seed(seed + 1)
    o = dict(d_z2=torch.randn(rows, D, generator=g), d_z1=torch.randn(rows, I, generator=g), d_hz=torch.randn(rows, D, generator=g),
             d_xres=torch.randn(rows, D, generator=g), d_ctx=torch.randn(rows, D, generator=g))
    for k in ('gFw', 'gFb', 'gAw', 'gAb'):
        o[k] = torch.randn(D, generator=g)
    return {k: v.cuda() for k, v in o.items()}


def run(A, t, o, rows, act_rows, res_rows, param_rows, I, act, passes):
    p = A.ops._p
    o = {k: v.clone() for k, v in o.items()}
    ops = torch.empty(A.LIB.query('acsr_dense_bwd_prep_floats', I), device='cuda')
    A.LIB.call('acsr_dense_bwd_prep', p(t['Wo']), p(t['W1']), p(t['W2']), D, I, p(ops), A.ops._stream())
    A.LIB.call('acsr_dense_bwd', p(t['d_out']), rows, act_rows, res_rows, param_rows, D, I, act, p(ops), p(t['z2']), p(t['b2']),
               p(t['h']), p(t['lnF_w']), p(t['st_f']), p(t['z1']), p(t['b1']), p(t['hz']), p(t['bo']), p(t['x_res']), p(t['lnA_w']),
               p(t['st_a']), t['p'], p(t['m_a']), p(t['m_f']), t['rng'].ptr if t['rng'] is not None else None, STREAM_A, STREAM_F,
               p(o['d_z2']), p(o['d_z1']), p(o['d_hz']), p(o['d_xres']), p(o['d_ctx']), p(o['gFw']), p(o['gFb']), p(o['gAw']),
               p(o['gAb']), passes, A.ops._stream())
    torch.cuda.synchronize()
    return o


def six_launches(A, t, o, rows, act_rows, res_rows, param_rows, I, act):
    """the six-launch chain the fused step runs where acsr_dense_bwd does not apply (inner sizes not a multiple of 64)"""
    p, st = A.ops._p, A.ops._stream()
    o = {k: v.clone() for k, v in o.items()}
    rngp = t['rng'].ptr if t['rng'] is not None else None
    d_h, d_a1 = torch.empty(rows, D, device='cuda'), torch.empty(rows, I, device='cuda')
    db = torch.zeros(3, max(I, D), device='cuda')
    A.LIB.call('acsr_bias_dropout_res_ln_bwd', p(t['d_out']), p(t['z2']), p(t['b2']), p(t['h']), p(t['lnF_w']), p(t['st_f']), rows, D,
               act_rows, act_rows, param_rows, t['p'], p(t['m_f']), rngp, STREAM_F, p(o['d_z2']), p(d_h), p(db[0]), p(o['gFw']),
               p(o['gFb']), st)
    A.ops.linear_tok(o['d_z2'], rows, D, t['W2'], I, d_a1, I, w_sn=1, w_sk=I, wkb=64 * I)
    A.LIB.call('acsr_bias_act_bwd', p(d_a1), p(t['z1']), p(t['b1']), rows, I, act, act_rows, param_rows, p(o['d_z1']), p(db[1]), st)
    A.ops.linear_tok(o['d_z1'], rows, I, t['W1'], D, d_h, D, w_sn=1, w_sk=D, wkb=64 * D, accumulate=True)
    A.LIB.call('acsr_bias_dropout_res_ln_bwd', p(d_h), p(t['hz']), p(t['bo']), p(t['x_res']), p(t['lnA_w']), p(t['st_a']), rows, D,
               act_rows, res_rows, param_rows, t['p'], p(t['m_a']), rngp, STREAM_A, p(o['d_hz']), p(o['d_xres']), p(db[2]),
               p(o['gAw']), p(o['gAb']), st)
    A.ops.linear_tok(o['d_hz'], rows, D, t['Wo'], D, o['d_ctx'], D, w_sn=1, w_sk=D, wkb=64 * D)
    torch.cuda.synchronize()
    return o


def check(o, o0, ref, rows, param_rows, rtol, what):
    for k in ('d_xres', 'd_ctx'):
        close(o[k], ref[k], rtol, '%s %s' % (what, k))
    for k in ('d_z2', 'd_z1', 'd_hz'):
        close(o[k][:param_rows], ref[k][:param_rows], rtol, '%s %s' % (what, k))
        assert torch.equal(o[k][param_rows:], o0[k][param_rows:]), '%s %s: rows past param_rows written' % (what, k)
    for k in ('gFw', 'gFb', 'gAw', 'gAb'):
        close(o[k] - o0[k], ref[k], rtol, '%s %s' % (what, k))


# (rows, act_rows, res_rows, param_rows): C2's first layer (both cotangent streams over T = 256 x 50 saved rows); the non-compact
# last layer (rows = act_rows = 2T, residual and parameters on T); ragged row counts (not multiples of the 128-row tile)
C2 = (25600, 12800, 12800, 12800)
CASES = [C2, (700, 700, 350, 350), (700, 350, 350, 350), (333, 333, 333, 100), (1000, 500, 250, 77)]


@pytest.mark.parametrize('rows,act_rows,res_rows,param_rows', CASES)
@pytest.mark.parametrize('mode', ['mask', 'philox', 'none'])
def test_dense_bwd_vs_fp64(A, rows, act_rows, res_rows, param_rows, mode):
    I, act = 256, 0
    seed = rows + act_rows + param_rows
    t, masks = make(A, rows, act_rows, res_rows, I, seed, mode)
    o0 = outputs(t, rows, I, seed)
    o = run(A, t, o0, rows, act_rows, res_rows, param_rows, I, act, 3)
    check(o, o0, reference(t, masks, rows, act_rows, res_rows, param_rows, act), rows, param_rows, 1e-4, mode)


@pytest.mark.parametrize('act', [0, 1, 2, 3, 4])
@pytest.mark.parametrize('I', [64, 128, 256])
@pytest.mark.parametrize('passes', [3, 1])
def test_dense_bwd_activations_widths_passes(A, act, I, passes):
    rows, act_rows, res_rows, param_rows = 700, 350, 350, 350
    seed = 100 * act + I + passes
    t, masks = make(A, rows, act_rows, res_rows, I, seed, 'mask')
    o0 = outputs(t, rows, I, seed)
    o = run(A, t, o0, rows, act_rows, res_rows, param_rows, I, act, passes)
    ref = reference(t, masks, rows, act_rows, res_rows, param_rows, act)
    check(o, o0, ref, rows, param_rows, 1e-4 if passes == 3 else 5e-3, 'act %d I %d passes %d' % (act, I, passes))


@pytest.mark.parametrize('rows,act_rows,res_rows,param_rows', CASES[:3])
@pytest.mark.parametrize('mode', ['mask', 'philox'])
def test_dense_bwd_vs_six_launches(A, rows, act_rows, res_rows, param_rows, mode):
    I, act = 256, 0
    seed = 3 * rows + act_rows
    t, _ = make(A, rows, act_rows, res_rows, I, seed, mode)
    o0 = outputs(t, rows, I, seed)
    o = run(A, t, o0, rows, act_rows, res_rows, param_rows, I, act, 3)
    old = six_launches(A, t, o0, rows, act_rows, res_rows, param_rows, I, act)
    ref = {k: v - o0[k] if k.startswith('g') else v for k, v in old.items()}
    check(o, o0, ref, rows, param_rows, 1e-4, 'six launches ' + mode)


def test_dense_bwd_philox_masks_are_the_forwards(A):
    """Philox draws (no mask tensors) give the same result as the forward's multipliers passed as explicit masks"""
    rows, act_rows, res_rows, param_rows, I = 1000, 500, 500, 500, 128
    t, masks = make(A, rows, act_rows, res_rows, I, 5, 'philox')
    o0 = outputs(t, rows, I, 5)
    o = run(A, t, o0, rows, act_rows, res_rows, param_rows, I, 0, 3)
    te = dict(t, m_f=masks[0].float().contiguous(), m_a=masks[1].float().contiguous(), rng=None)
    oe = run(A, te, o0, rows, act_rows, res_rows, param_rows, I, 0, 3)
    for k in o:
        close(o[k], oe[k], 1e-6, k)


def test_dense_bwd_rejects_bad_arguments(A):
    rows, I = 256, 128
    t, _ = make(A, rows, rows, rows, I, 9, 'mask')
    o0 = outputs(t, rows, I, 9)
    o = {k: v.clone() for k, v in o0.items()}
    p = A.ops._p
    ops = torch.zeros(A.LIB.query('acsr_dense_bwd_prep_floats', I), device='cuda')

    def rc(**kw):
        a = dict(d_out=p(t['d_out']), rows=rows, act_rows=rows, res_rows=rows, param_rows=rows, d=D, I=I, act=0, ops=p(ops),
                 z2=p(t['z2']), b2=p(t['b2']), h=p(t['h']), lnF_w=p(t['lnF_w']), st_f=p(t['st_f']), z1=p(t['z1']), b1=p(t['b1']),
                 hz=p(t['hz']), bo=p(t['bo']), x_res=p(t['x_res']), lnA_w=p(t['lnA_w']), st_a=p(t['st_a']), p_drop=P_DROP,
                 m_a=p(t['m_a']), m_f=p(t['m_f']), rng=None, sa=STREAM_A, sf=STREAM_F, d_z2=p(o['d_z2']), d_z1=p(o['d_z1']),
                 d_hz=p(o['d_hz']), d_xres=p(o['d_xres']), d_ctx=p(o['d_ctx']), gFw=p(o['gFw']), gFb=p(o['gFb']), gAw=p(o['gAw']),
                 gAb=p(o['gAb']), passes=3)
        a.update(kw)
        return A.LIB.query('acsr_dense_bwd', *a.values(), A.ops._stream())
    assert rc(d=128) == -2                               # hidden size other than 64
    assert rc(I=96) == -2 and rc(I=320) == -2 and rc(I=0) == -2
    for k in ('d_out', 'ops', 'z2', 'z1', 'st_a', 'x_res', 'd_z1', 'd_xres', 'd_ctx', 'gAb'):
        assert rc(**{k: None}) == -1, k
    assert rc(m_a=None) == -1                            # p > 0 without a mask or the device RNG
    assert rc(param_rows=rows + 1) == -1
    assert rc(act_rows=0) == -1 and rc(res_rows=0) == -1
    assert rc(act=5) == -1
    assert rc(passes=2) == -1
    assert A.LIB.query('acsr_dense_bwd_prep', p(t['Wo']), p(t['W1']), p(t['W2']), D, 100, p(ops), A.ops._stream()) == -2
    assert A.LIB.query('acsr_dense_bwd_prep_floats', 100) == 0
    torch.cuda.synchronize()
    for k in o:
        assert torch.equal(o[k], o0[k]), k                # nothing launched
