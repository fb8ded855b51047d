"""General tcgen05 GEMM (acsr_gemm_batch, gemm_ks.cu) against fp64 matmuls: every operand form the encoder
uses (forward, transposed weight, K-concatenated inputs, token-axis contraction for weight gradients), every
epilogue, ragged sizes, hidden sizes 64 / 128 / 256, multi-problem launches.  3xTF32 -> fp32-level accuracy."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import acsr_oracle as O


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


def rnd(g, *shape, s=1.0):
    return (torch.randn(*shape, generator=g) * s).cuda()


@pytest.mark.parametrize('M,N,K,accumulate', [(300, 64, 64, False), (1280, 256, 64, False), (257, 128, 128, True), (1000, 50, 64, False),
                                              (700, 64, 50, True), (513, 320, 96, False), (640, 1024, 256, False), (384, 256, 1024, True),
                                              (129, 16, 8, False), (5, 4, 4, False)])
def test_gemm_store(A, M, N, K, accumulate):
    g = torch.Generator().manual_seed(M + N + K)
    X, W, b, Y0 = rnd(g, M, K), rnd(g, N, K, s=0.2), rnd(g, N), rnd(g, M, N)
    Y = Y0.clone()
    A.ops.gemm_batch([A.ops.gemm_problem(X, W, Y, M, N, K, bias=b, accumulate=accumulate)])
    ref = X.double() @ W.double().t() + b.double() + (Y0.double() if accumulate else 0)
    # the tensor core truncates when it accumulates: the error grows with the length of the MMA chain (3 passes x K/8 MMAs)
    close(Y, ref, 3e-6 if K <= 256 else 2e-5, 'store')


def test_gemm_operand_forms(A):
    g = torch.Generator().manual_seed(5)
    T2, d, I, L = 700, 128, 64, 50
    ops = A.ops
    # input gradient through W2 [d, I]: d_a1 = d_z2 . W2  (weight read transposed: element (n, k) = W2[k, n])
    dz2, W2 = rnd(g, T2, d), rnd(g, d, I, s=0.1)
    da1 = torch.empty(T2, I).cuda()
    ops.gemm_batch([ops.gemm_problem(dz2, W2, da1, T2, I, d, b_strides=(1, I, 0, d))])
    close(da1, dz2.double() @ W2.double(), 3e-6, 'transposed weight')
    # K-concatenated stacked inputs: d_x += sum_b d_qkv[b] . Wqkv[b]
    dqkv, Wqkv, dx0 = rnd(g, 3, T2, d), rnd(g, 3, d, d, s=0.1), rnd(g, T2, d)
    dx = dx0.clone()
    ops.gemm_batch([ops.gemm_problem(dqkv, Wqkv, dx, T2, d, 3 * d, a_strides=(d, 1, T2 * d, d), b_strides=(1, d, d * d, d), accumulate=True)])
    ref = dx0.double() + sum(dqkv[i].double() @ Wqkv[i].double() for i in range(3))
    close(dx, ref, 3e-6, 'K-concat')
    # a leading sub-range of rows only
    dx2 = dx0.clone()
    ops.gemm_batch([ops.gemm_problem(dqkv, Wqkv, dx2, 300, d, 3 * d, a_strides=(d, 1, T2 * d, d), b_strides=(1, d, d * d, d), accumulate=True)])
    close(dx2[:300], ref[:300], 3e-6, 'K-concat rows')
    assert torch.equal(dx2[300:], dx0[300:])
    # gate: N = L = 50 forward with bias, K = L = 50 input gradient (unaligned rows)
    x, Wg, bg = rnd(g, T2, d), rnd(g, L, d, s=0.1), rnd(g, L)
    gl = torch.empty(T2, L).cuda()
    dgl, dmq0 = rnd(g, T2, L), rnd(g, T2, d)
    dmq = dmq0.clone()
    ops.gemm_batch([ops.gemm_problem(x, Wg, gl, T2, L, d, bias=bg),
                    ops.gemm_problem(dgl, Wg, dmq, T2, d, L, b_strides=(1, d, 0, L), accumulate=True)])
    close(gl, x.double() @ Wg.double().t() + bg.double(), 3e-6, 'gate fwd')
    close(dmq, dmq0.double() + dgl.double() @ Wg.double(), 3e-6, 'gate dgrad')
    # five projections that read the same input, one launch, outputs in one stacked buffer
    W5, b5 = rnd(g, 5, d, d, s=0.1), rnd(g, 5, d)
    y5 = torch.empty(5, T2, d).cuda()
    ops.gemm_batch([ops.gemm_problem(x, W5[i], y5[i], T2, d, d, bias=b5[i]) for i in range(5)])
    for i in range(5):
        close(y5[i], x.double() @ W5[i].double().t() + b5[i].double(), 3e-6, 'proj %d' % i)
    # strided output (ldc > N)
    wide = torch.zeros(T2, 3 * d).cuda()
    ops.gemm_batch([ops.gemm_problem(x, W5[0], wide[:, d:], T2, d, d, ldc=3 * d)])
    close(wide[:, d:2 * d], x.double() @ W5[0].double().t(), 3e-6, 'ldc')
    assert float(wide[:, :d].abs().max()) == 0.0 and float(wide[:, 2 * d:].abs().max()) == 0.0


@pytest.mark.parametrize('T,N,K,bias,splits', [(12800, 64, 64, True, 0), (1000, 256, 64, True, 0), (777, 64, 256, False, 3), (3000, 50, 128, True, 0),
                                               (2500, 128, 128, True, 1), (4096, 1024, 256, True, 0), (333, 256, 1024, False, 0)])
def test_gemm_wgrad(A, T, N, K, bias, splits):
    """dW[N,K] += dY^T.X over the token axis (split-K + atomics), db = column sums of dY."""
    g = torch.Generator().manual_seed(T + N + K)
    dY, X = rnd(g, T, N), rnd(g, T, K)
    dW0 = rnd(g, N, K)
    db0 = rnd(g, N)
    dW, db = dW0.clone(), db0.clone()
    A.ops.gemm_batch([A.ops.wgrad_problem(dY, X, T, N, K, dW, db if bias else None, k_splits=splits)])
    close(dW - dW0, dY.double().t() @ X.double(), 1e-5, 'dW')
    if bias:
        close(db - db0, dY.double().sum(0), 1e-5, 'db')
    else:
        assert torch.equal(db, db0)


def test_gemm_wgrad_row_subrange_and_batch(A):
    """a layer's weight gradients in ONE launch: different shapes, row sub-ranges (stream halves) of wider buffers."""
    g = torch.Generator().manual_seed(11)
    T, d, I, L = 1500, 64, 256, 50
    ops = A.ops
    d_z2, a1, d_z1, h, d_gl, mq = rnd(g, 2 * T, d), rnd(g, T, I), rnd(g, 2 * T, I), rnd(g, T, d), rnd(g, 2 * T, L), rnd(g, T, d)
    dW2, dW1, dWg, dbg = (torch.zeros(s).cuda() for s in ((d, I), (I, d), (L, d), (L,)))
    ops.gemm_batch([ops.wgrad_problem(d_z2, a1, T, d, I, dW2), ops.wgrad_problem(d_z1, h, T, I, d, dW1),
                    ops.wgrad_problem(d_gl[T:], mq, T, L, d, dWg, dbg)])
    close(dW2, d_z2[:T].double().t() @ a1.double(), 1e-5, 'dW2')
    close(dW1, d_z1[:T].double().t() @ h.double(), 1e-5, 'dW1')
    close(dWg, d_gl[T:].double().t() @ mq.double(), 1e-5, 'dWg')
    close(dbg, d_gl[T:].double().sum(0), 1e-5, 'dbg')


@pytest.mark.parametrize('act', ['gelu', 'relu', 'swish', 'tanh', 'sigmoid'])
@pytest.mark.parametrize('d,I', [(64, 256), (128, 64), (256, 1024)])
def test_gemm_act(A, act, d, I):
    g = torch.Generator().manual_seed(9)
    R = 1100
    X, W, b = rnd(g, R, d), rnd(g, I, d, s=0.2), rnd(g, I)
    Z, A1 = torch.empty(R, I).cuda(), torch.empty(R, I).cuda()
    A.ops.gemm_batch([A.ops.gemm_problem(X, W, Z, R, I, d, bias=b, epilogue=A.ops.EPI_ACT, act=A.ops.ACT_IDS[act], C2=A1)])
    zr = X.double() @ W.double().t()
    close(Z, zr, 3e-6 if d <= 256 else 2e-5, 'Z')
    # activations with slope <= ~1.1: the output error is bounded by the input error (relative to max |z|, not max |act|).
    # The reference is evaluated in float64: a float32 evaluation of erf on the host has been off by 4e-4, beyond the bound.
    ref = O.act_fn(act)((zr + b.double()).cpu())
    err = float((A1.double().cpu() - ref).abs().max())
    assert err <= 1e-5 * float(ref.abs().max()) + 4e-6 * float(zr.abs().max()), (err, float(zr.abs().max()))


@pytest.mark.parametrize('d,K,p,explicit', [(64, 64, 0.0, False), (64, 256, 0.5, True), (128, 128, 0.5, True), (128, 64, 0.5, False),
                                            (256, 256, 0.3, True), (256, 1024, 0.5, False), (32, 32, 0.5, True)])
def test_gemm_bdrl(A, d, K, p, explicit):
    g = torch.Generator().manual_seed(d + K + int(p * 10))
    R, Tres = 2 * 450, 450
    X, W, b, res = rnd(g, R, K), rnd(g, d, K, s=0.2), rnd(g, d), rnd(g, Tres, d)
    lw, lb = rnd(g, d), rnd(g, d)
    mask = ((torch.rand(R, d, generator=g) >= p).float() / (1 - p)).cuda() if explicit else None
    rng = A.ops.DeviceRng(77, torch.device('cuda'))
    HZ, out, stats = torch.empty(R, d).cuda(), torch.empty(R, d).cuda(), torch.empty(R, 2).cuda()
    A.ops.gemm_batch([A.ops.gemm_problem(X, W, HZ, R, d, K, bias=b, epilogue=A.ops.EPI_BDRL, res=res, res_rows=Tres, ln_w=lw, ln_b=lb,
                                         eps=1e-12, p_drop=p, mask=mask, rngp=rng.ptr, rng_stream=19, out=out, stats=stats)])
    hz = X.double() @ W.double().t()
    close(HZ, hz, 3e-6 if K <= 256 else 2e-5, 'HZ')
    # the unfused row-wise kernel with the same rng / mask is the reference of the epilogue (same Philox counters)
    out2, stats2 = torch.empty(R, d).cuda(), torch.empty(R, 2).cuda()
    A.LIB.call('acsr_bias_dropout_res_ln_fwd', HZ.data_ptr(), b.data_ptr(), res.data_ptr(), lw.data_ptr(), lb.data_ptr(), 1e-12,
               R, d, Tres, p, mask.data_ptr() if explicit else None, rng.ptr, 19, out2.data_ptr(), stats2.data_ptr(), A.ops._stream())
    close(out, out2, 2e-5, 'out vs unfused')
    close(stats, stats2, 2e-5, 'stats vs unfused')
    if explicit or p == 0.0:
        m = mask.double() if explicit else 1.0
        x = (hz + b.double()) * m + res.double().repeat(R // Tres, 1)
        mean = x.mean(-1, keepdim=True)
        var = ((x - mean) ** 2).mean(-1, keepdim=True)
        close(out, (x - mean) / torch.sqrt(var + 1e-12) * lw.double() + lb.double(), 2e-5, 'out')


def test_gemm_many_tiles_persistent(A):
    """more work items than SMs: every CTA walks several (m-tile, n-block) items through both accumulator stages."""
    g = torch.Generator().manual_seed(3)
    M, N, K = 128 * 330 + 17, 192, 160
    X, W = rnd(g, M, K), rnd(g, N, K, s=0.1)
    Y = torch.empty(M, N).cuda()
    A.ops.gemm_batch([A.ops.gemm_problem(X, W, Y, M, N, K)])
    close(Y, X.double() @ W.double().t(), 3e-6, 'persistent')


def test_gemm_single_pass_tf32(A):
    g = torch.Generator().manual_seed(4)
    M, N, K = 512, 128, 128
    X, W = rnd(g, M, K), rnd(g, N, K, s=0.1)
    Y = torch.empty(M, N).cuda()
    A.ops.gemm_batch([A.ops.gemm_problem(X, W, Y, M, N, K)], passes=1)
    close(Y, X.double() @ W.double().t(), 2e-3, 'tf32')


def test_gemm_rejects_bad_arguments(A):
    x = torch.zeros(8, 8).cuda()
    with pytest.raises(A.AcsrError):
        A.ops.gemm_batch([A.ops.gemm_problem(x, x, x, 8, 8, 8)], passes=2)
    with pytest.raises(A.AcsrError):      # LayerNorm epilogue wider than one CTA's accumulator
        big = torch.zeros(8, 512).cuda()
        A.ops.gemm_batch([A.ops.gemm_problem(x, torch.zeros(512, 8).cuda(), big, 8, 512, 8, epilogue=A.ops.EPI_BDRL, res=big, res_rows=8,
                                             ln_w=big, ln_b=big, out=big, stats=big)])
    with pytest.raises(A.AcsrError):
        A.ops.gemm_problem(torch.zeros(8, 8), x, x, 8, 8, 8)
