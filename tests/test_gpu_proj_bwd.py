"""acsr_proj_input_grad: the input gradient of a layer's projections in one launch, against a float64 restatement of the chain
it replaces (d_qkv[0:2] += d_aqk.Waqk ; d_mq += d_gl.Wg ; d_x += [d_mq d_mk d_mv].[Wq; Wk; Wv]) and against that chain run as
three acsr_linear_tok launches.  Tolerances as the linear_tok tests: 3e-6 of the tensor's max |value| for 3xTF32."""
import pytest
import torch

pytestmark = pytest.mark.gpu

D = 64


@pytest.fixture(scope='module')
def A():
    import ac_tsr_b200 as pkg
    pkg.LIB.load()
    return pkg


def close(a, b, rtol, what=''):
    a = a.detach().double().cpu()
    b = b.detach().double().cpu()
    scale = float(b.abs().max().clamp(min=1e-30))
    err = float((a - b).abs().max())
    assert err <= rtol * scale + 1e-12, '%s: err %.3e scale %.3e' % (what, err, scale)


def make(T2, L, gate, seed):
    g = torch.Generator().manual_seed(seed)
    t = dict(d_qkv=torch.randn(3, T2, D, generator=g), d_aqk=torch.randn(2, T2, D, generator=g),
             d_gl=torch.randn(T2, L, generator=g) if gate else None, Wqkv=torch.randn(3, D, D, generator=g) * 0.1,
             Waqk=torch.randn(2, D, D, generator=g) * 0.1, Wg=torch.randn(L, D, generator=g) * 0.1 if gate else None,
             d_x=torch.randn(T2, D, generator=g))
    return {k: (None if v is None else v.cuda()) for k, v in t.items()}


def reference(t, rows):
    dq = t['d_qkv'].double().clone()
    for i in range(2):
        dq[i] += t['d_aqk'][i].double() @ t['Waqk'][i].double()
    if t['d_gl'] is not None:
        dq[0] += t['d_gl'].double() @ t['Wg'].double()
    dx = t['d_x'].double().clone()
    dx[:rows] += sum(dq[i, :rows] @ t['Wqkv'][i].double() for i in range(3))
    return dq, dx


def run(A, t, rows, keep, passes, L):
    d_qkv, d_x = t['d_qkv'].clone(), t['d_x'].clone()
    p = A.ops._p
    A.LIB.call('acsr_proj_input_grad', p(d_qkv), p(t['d_aqk']), d_qkv.shape[1], p(t['d_gl']), L, p(t['Wqkv']), p(t['Waqk']),
               p(t['Wg']), D, rows, keep, p(d_x), passes, A.ops._stream())
    torch.cuda.synchronize()
    return d_qkv, d_x


def old_chain(A, t, rows, L):
    """the three acsr_linear_tok launches of the fused step before acsr_proj_input_grad"""
    d_qkv, d_x = t['d_qkv'].clone(), t['d_x'].clone()
    T2 = d_qkv.shape[1]
    A.ops.linear_tok(t['d_aqk'], T2, D, t['Waqk'], D, d_qkv, D, w_sn=1, w_sk=D, wkb=64 * D, accumulate=True,
                     batch=2, sx=T2 * D, sw=D * D, sb=0, sy=T2 * D)
    if t['d_gl'] is not None:
        A.ops.linear_tok(t['d_gl'], T2, L, t['Wg'], D, d_qkv[0], D, ldx=L, w_sn=1, w_sk=D, wkb=64 * D, accumulate=True)
    A.ops.linear_tok(d_qkv, rows, 3 * D, t['Wqkv'], D, d_x, D, ldx=D, xkb=T2 * D, w_sn=1, w_sk=D, wkb=D * D, accumulate=True)
    torch.cuda.synchronize()
    return d_qkv, d_x


# (T2, rows, rows_keep): C2's last layer (rows = 2T) and first layer (rows = T) at T = 256 x 50; a ragged batch of 7 x 50
CASES = [(25600, 25600, 12800), (25600, 12800, 12800), (700, 700, 350), (700, 350, 350), (700, 333, 100)]


@pytest.mark.parametrize('T2,rows,keep', CASES)
@pytest.mark.parametrize('gate', [True, False])
@pytest.mark.parametrize('passes', [3, 1])
def test_proj_input_grad_vs_fp64(A, T2, rows, keep, gate, passes):
    L = 50
    t = make(T2, L, gate, seed=T2 + rows + keep + int(gate))
    d_qkv, d_x = run(A, t, rows, keep, passes, L)
    dq, dx = reference(t, rows)
    rtol = 3e-6 if passes == 3 else 2e-3          # one TF32 product: 10-bit mantissa operands
    close(d_x[:rows], dx[:rows], rtol, 'd_x')
    assert torch.equal(d_x[rows:], t['d_x'][rows:])
    for i, name in ((0, 'd_mq'), (1, 'd_mk')):
        close(d_qkv[i, :keep], dq[i, :keep], rtol, name)
        assert torch.equal(d_qkv[i, keep:], t['d_qkv'][i, keep:]), name + ' rows past rows_keep'
    assert torch.equal(d_qkv[2], t['d_qkv'][2])


@pytest.mark.parametrize('T2,rows,keep', CASES[:3])
@pytest.mark.parametrize('gate', [True, False])
def test_proj_input_grad_vs_linear_tok_chain(A, T2, rows, keep, gate):
    L = 50
    t = make(T2, L, gate, seed=7 * T2 + rows)
    d_qkv, d_x = run(A, t, rows, keep, 3, L)
    o_qkv, o_x = old_chain(A, t, rows, L)
    close(d_x[:rows], o_x[:rows], 3e-6, 'd_x')
    close(d_qkv[:2, :keep], o_qkv[:2, :keep], 3e-6, 'd_mq / d_mk')


def test_proj_input_grad_gate_widths(A):
    for L in (1, 8, 64):
        t = make(300, L, True, seed=L)
        d_qkv, d_x = run(A, t, 300, 300, 3, L)
        dq, dx = reference(t, 300)
        close(d_x, dx, 3e-6, 'd_x L=%d' % L)
        close(d_qkv[0], dq[0], 3e-6, 'd_mq L=%d' % L)


def test_proj_input_grad_rejects_bad_arguments(A):
    t = make(256, 50, True, seed=1)
    p = A.ops._p
    d_qkv, d_x = t['d_qkv'].clone(), t['d_x'].clone()

    def rc(**kw):
        a = dict(d_qkv=p(d_qkv), d_aqk=p(t['d_aqk']), plane=256, d_gl=p(t['d_gl']), L=50, Wqkv=p(t['Wqkv']), Waqk=p(t['Waqk']),
                 Wg=p(t['Wg']), d=D, rows=256, keep=128, d_x=p(d_x), passes=3)
        a.update(kw)
        return A.LIB.query('acsr_proj_input_grad', *a.values(), A.ops._stream())
    assert rc(d_qkv=None) == -1
    assert rc(d_aqk=None) == -1
    assert rc(Wqkv=None) == -1
    assert rc(d_x=None) == -1
    assert rc(Wg=None) == -1                       # d_gl without Wg
    assert rc(keep=257) == -1                      # rows_keep > rows
    assert rc(rows=257, keep=0) == -1              # rows > plane
    assert rc(L=65) == -1 and rc(L=0) == -1        # gate width out of range
    assert rc(d=128) == -2                         # hidden size other than 64
    assert rc(passes=2) == -1
    torch.cuda.synchronize()
    assert torch.equal(d_qkv, t['d_qkv']) and torch.equal(d_x, t['d_x'])
    assert rc(d_gl=None, Wg=None, L=0) == 0        # without the gate L is ignored
    torch.cuda.synchronize()
