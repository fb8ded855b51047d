"""Micro-benchmark of the encoder GEMM shapes: tcgen05 token-tile kernel vs the library GEMM (CUDA-graph replay)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import __graft_entry__ as ge
ge.build()
import ac_tsr_b200 as A
from ac_tsr_b200 import ops

dev = torch.device('cuda')


def bench(f, iters=20):
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        for _ in range(3):
            f()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            for _ in range(iters):
                f()
        g.replay()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3


T, d, I, L = 12800, 64, 256, 50
for rows in (T, 2 * T):
    x = torch.randn(rows, d, device=dev)
    W = torch.randn(d, d, device=dev) * .1
    W1 = torch.randn(I, d, device=dev) * .1
    W2 = torch.randn(d, I, device=dev) * .1
    b = torch.randn(d, device=dev)
    y = torch.empty(rows, d, device=dev)
    z1, a1 = torch.empty(rows, I, device=dev), torch.empty(rows, I, device=dev)
    a1.normal_()
    res = torch.randn(T, d, device=dev)
    out, stats = torch.empty(rows, d, device=dev), torch.empty(rows, 2, device=dev)
    lw, lb = torch.ones(d, device=dev), torch.zeros(d, device=dev)
    rng = ops.DeviceRng(1, dev)
    print('rows %d' % rows)
    print('  64->64    tok %.1f  | addmm %.1f' % (bench(lambda: ops.linear_tok(x, rows, d, W, d, y, d, bias=b)), bench(lambda: torch.addmm(b, x, W.t(), out=y))))
    print('  64->64 acc tok %.1f | addmm_ %.1f' % (bench(lambda: ops.linear_tok(x, rows, d, W, d, y, d, w_sn=1, w_sk=d, wkb=64 * d, accumulate=True)), bench(lambda: y.addmm_(x, W))))
    print('  64->256   tok %.1f  | mm %.1f' % (bench(lambda: ops.linear_tok(x, rows, d, W1, I, z1, I)), bench(lambda: torch.mm(x, W1.t(), out=z1))))
    print('  256->64   tok %.1f  | mm %.1f' % (bench(lambda: ops.linear_tok(a1, rows, I, W2, d, y, d)), bench(lambda: torch.mm(a1, W2.t(), out=y))))
    print('  64->64 +bdrl fused %.1f | tok + bdrl %.1f' % (
        bench(lambda: ops.linear_tok_bdrl(x, rows, d, W, b, res, T, lw, lb, 1e-12, 0.5, None, rng.ptr, 3, y, out, stats)),
        bench(lambda: (ops.linear_tok(x, rows, d, W, d, y, d), A.LIB.call('acsr_bias_dropout_res_ln_fwd', y.data_ptr(), b.data_ptr(), res.data_ptr(), lw.data_ptr(), lb.data_ptr(), 1e-12, rows, d, T, 0.5, None, rng.ptr, 3, out.data_ptr(), stats.data_ptr(), ops._stream())))))
x = torch.randn(T, d, device=dev)
Wqkv = torch.randn(3, d, d, device=dev) * .1
bq = torch.randn(3, 1, d, device=dev)
qkv = torch.empty(3, T, d, device=dev)
print('QKV batch3 tok %.1f | baddbmm %.1f' % (bench(lambda: ops.linear_tok(x, T, d, Wqkv, d, qkv, d, bias=bq, batch=3, sx=0, sw=d * d, sb=d, sy=T * d)),
                                              bench(lambda: torch.baddbmm(bq, x.unsqueeze(0).expand(3, T, d), Wqkv.transpose(1, 2), out=qkv))))
dq = torch.randn(3, 2 * T, d, device=dev)
dx = torch.randn(2 * T, d, device=dev)
print('d_x K=192 tok %.1f | 3x addmm_ %.1f' % (bench(lambda: ops.linear_tok(dq, 2 * T, 3 * d, Wqkv, d, dx, d, ldx=d, xkb=2 * T * d, w_sn=1, w_sk=d, wkb=d * d, accumulate=True)),
                                               bench(lambda: [dx.addmm_(dq[i], Wqkv[i]) for i in range(3)])))
V, B = 12102, 256
Gt = torch.randn(V, 2 * B, device=dev)
o2 = torch.randn(2 * B, d, device=dev)
dE = torch.zeros(V, d, device=dev)
print('dE tok %.1f | addmm_ %.1f' % (bench(lambda: ops.linear_tok(Gt, V, B, o2, d, dE, d, ldx=2 * B, w_sn=1, w_sk=d, wkb=64 * d, accumulate=True)),
                                     bench(lambda: dE.addmm_(Gt[:, :B], o2[:B]))))
