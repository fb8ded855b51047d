"""gloo tests (CPU, world size 2 and 3) of the gradient-clip norm over a vocab-sharded item table (FlatAdam.set_table_shard): with
a torch restatement of the local norm kernel injected, the partial of the replicated parameters plus the all-gathered partials of
every rank's table shard must give the norm of the full gradient in the reference layout, and every rank the same coefficient.
Also: which `clip_grad_norm` settings the device clip takes is decided from the setting alone."""
import os
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def torch_partial(grad, q, ranges=None, out=None, work=None):
    """acsr_grad_norm_partial restated: sum |g|^q (max |g| for q = inf) over the ranges, in fp64"""
    ranges = [(0, grad.numel())] if ranges is None else ranges
    g = torch.cat([grad[b:e] for b, e in ranges]).double().abs()
    v = g.max() if q == float('inf') else (g ** q).sum()
    out.copy_(v.reshape(1) if g.numel() else torch.zeros(1, dtype=torch.float64))
    return out


def combine(parts, q):
    """acsr_adam_step_clipped's total and coefficient, restated: partials in index order, the q-th root, torch's clamp"""
    s = parts[0].clone()
    for p in parts[1:]:
        s = torch.maximum(s, p) if q == float('inf') else s + p
    total = (s if q == float('inf') else s ** (1.0 / q)).float()
    return total, torch.clamp(0.5 / (total + 1e-6), max=1.0)


class Net(torch.nn.Module):
    def __init__(self, V, d):
        super().__init__()
        self.lin = torch.nn.Linear(d, 2 * d)
        self.item_embedding = torch.nn.Embedding(V, d)
        self.norm = torch.nn.LayerNorm(d)


def _worker(rank, world, port, V, q, ret):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        import ac_tsr_b200 as A
        d = 12
        torch.manual_seed(0)
        net = Net(V, d)
        full_grads = {n: torch.randn_like(p) * (1 + i) for i, (n, p) in enumerate(net.named_parameters())}
        full_grads['item_embedding.weight'][5] *= 40.0                  # one large table row: the inf-norm sits in the table
        vp = A.dist.VocabParallel(V, compute=object(), align=8, sharded=True)
        net.item_embedding.weight = torch.nn.Parameter(vp.make_shard(net.item_embedding.weight.detach()))
        opt = A.FlatAdam(net, 1e-3, clip=A.FlatAdam.device_clip({'max_norm': 0.5, 'norm_type': q}))
        opt._norm_partial = torch_partial
        E = net.item_embedding.weight
        opt.set_table_shard(E, (vp.hi - vp.lo) * d, vp._all_gather)
        with torch.no_grad():
            for n, p in net.named_parameters():
                if p is E:                                          # the owner's rows; the padded rows keep their zero gradient
                    p.grad[:vp.hi - vp.lo].copy_(full_grads[n][vp.lo:vp.hi])
                else:                                              # replicated (all-reduced) parameters: the same on every rank
                    p.grad.copy_(full_grads[n])
        parts = opt._clip_partials()
        assert parts.shape == (1 + world,)
        total, coef = combine(parts, float(q))
        want = torch.linalg.vector_norm(torch.cat([g.reshape(-1) for g in full_grads.values()]).double(), float(q))
        assert abs(float(total) - float(want)) <= 1e-6 * float(want), (float(total), float(want))
        assert float(coef) < 1.0
        # the full table gradient gathered back to the reference layout has the same norm as the shards' partials say
        assert torch.equal(vp.gather_full(E.grad), full_grads['item_embedding.weight'])
        # every rank sees the same partials in the same order, hence bit for bit the same coefficient
        got = vp._all_gather(torch.cat((parts, coef.double().reshape(1))))
        for r in range(world):
            assert torch.equal(got[r], got[0]), (rank, got)
        ret[rank] = 'ok'
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize('world,V', [(2, 97), (3, 40)])
@pytest.mark.parametrize('q', [2, 'inf'])
def test_sharded_clip_norm_equals_the_full_gradient_norm(world, V, q):
    mgr = mp.Manager()
    ret = mgr.dict()
    port = 29300 + (os.getpid() + V + world) % 250
    mp.spawn(_worker, args=(world, port, V, q, ret), nprocs=world, join=True)
    assert dict(ret) == {r: 'ok' for r in range(world)}


def test_device_clip_is_decided_from_the_setting_alone():
    import ac_tsr_b200 as A
    dc = A.FlatAdam.device_clip
    assert dc({'max_norm': 0.5, 'norm_type': 2}) == (0.5, 2.0)
    assert dc({'max_norm': 5}) == (5.0, 2.0)                                          # torch's default norm_type
    assert dc({'max_norm': 1, 'norm_type': 'inf'}) == (1.0, float('inf'))
    assert dc({'max_norm': 1, 'norm_type': float('inf')}) == (1.0, float('inf'))
    assert dc({'max_norm': 1, 'norm_type': 3.5}) == (1.0, 3.5)
    for torch_only in (None, {}, {'norm_type': 2}, {'max_norm': 1, 'error_if_nonfinite': True}, {'max_norm': 1, 'foreach': None},
                       {'max_norm': 1, 'norm_type': 0}, {'max_norm': 1, 'norm_type': -1}, {'max_norm': 0}, {'max_norm': -1},
                       {'max_norm': 1, 'norm_type': 'nan'}, {'max_norm': 'x'}, {'max_norm': 1, 'norm_type': '-inf'}):
        assert dc(torch_only) is None, torch_only
