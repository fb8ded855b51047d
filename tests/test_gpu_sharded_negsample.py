"""Sampled ranking and BPR over a vocab-sharded item table on the GPU: the shard kernels of negsample.cu / bpr.cu summed over W
row ranges against the unsharded kernels (scores, hit flags, counts, row_x and losses bit-identical; d_out and the table
gradient up to the order of the atomics), their argument checks, and the real VocabParallel with the CUDA kernels over gloo."""
import json
import os
import sys
import time

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


@pytest.fixture(scope='module')
def A():
    import ac_tsr_b200 as pkg
    pkg.LIB.load()
    return pkg


def ranges(V, W):
    per = (V + W - 1) // W
    return [(r * per, min(V, (r + 1) * per)) for r in range(W)]


def make_cand(V, M, N, bounds, g):
    """candidates with duplicates, the positive among the negatives, id 0, out-of-range ids and every shard boundary"""
    cand = torch.randint(1, V, (M, N + 1), generator=g)
    edge = sorted({0, V - 1, -5, V + 3} | {i for lo, hi in bounds for i in (lo - 1, lo, hi - 1, hi) if 0 <= i < V})
    e = torch.tensor(edge)
    if N >= 1:
        cand[::2, 1] = cand[::2, 0]                                    # the positive again
    if N >= 1 + e.numel():
        cand[:, 2:2 + e.numel()] = e
    if N >= 8:
        cand[:, -4:] = cand[:, -5:-4]                                  # duplicates
    cand[1::3, 0] = e[torch.arange(cand[1::3].shape[0]) % e.numel()]
    return cand


@pytest.mark.parametrize('W', [2, 3, 8])
@pytest.mark.parametrize('d', [32, 64, 128, 256])
@pytest.mark.parametrize('N', [1, 99, 1000])
def test_shard_kernels_sum_to_unsharded(A, W, d, N):
    ops, LIB = A.ops, A.LIB
    g = torch.Generator().manual_seed(W * 1000 + d + N)
    V, M, k = 5003, 96, 50
    bounds = ranges(V, W)
    E = (torch.randn(V, d, generator=g) * 0.2).cuda()
    out = torch.randn(M, d, generator=g).cuda()
    out[5] = 0                                                         # every candidate ties with the positive
    cand = make_cand(V, M, N, bounds, g).cuda()
    shards = [E[lo:hi].clone() for lo, hi in bounds]                   # each rank's own storage
    # ---- sampled ranking ----
    rec0, s0, cnt0 = ops.candidate_rank(out, E, cand, k, want_scores=True, want_counts=True)
    rec1, _ = ops.candidate_rank(out, E, cand, k)
    tot = torch.zeros_like(s0)
    for (lo, hi), sh in zip(bounds, shards):
        tot += ops.candidate_scores_shard(out, sh, lo, hi, V, cand)
    assert torch.equal(tot, s0)
    rec, cnt = ops.candidate_rank_scores(tot, cand, V, k, want_counts=True)
    assert torch.equal(rec, rec0) and torch.equal(cnt, cnt0)
    rec2, none = ops.candidate_rank_scores(tot, cand, V, k)
    assert none is None and torch.equal(rec2, rec1)
    # ---- BPR: [calibrated ; attacked] rows, the first half trains the table ----
    M2 = 2 * M
    o2 = torch.randn(M2, d, generator=g).cuda()
    pos = torch.randint(1, V, (M2,), generator=g)
    neg = torch.randint(1, V, (M2,), generator=g)
    edge = torch.tensor(sorted({i for lo, hi in bounds for i in (lo - 1, lo, hi - 1) if 0 <= i < V}))
    pos[:edge.numel()] = edge
    neg[1:edge.numel() + 1] = edge
    neg[::7] = pos[::7]
    pos[3] = 0
    pos, neg = pos.cuda(), neg.cuda()
    gamma = 1e-10
    row_x0, row_loss0, loss0 = (torch.empty(M2, device='cuda'), torch.empty(M2, device='cuda'), torch.empty(2, device='cuda'))
    LIB.call('acsr_bpr_loss_fwd', ops._p(o2), ops._p(E), ops._p(pos, torch.int64), ops._p(neg, torch.int64), M2, d, 2, gamma,
             ops._p(row_x0), ops._p(row_loss0), ops._p(loss0), ops._stream())
    dots = torch.zeros((M2, 2), device='cuda')
    for (lo, hi), sh in zip(bounds, shards):
        dots += ops.bpr_dots_shard(o2, sh, lo, hi, V, pos, neg)
    loss, row_x = ops.bpr_loss_from_dots(dots, 2, gamma)
    assert torch.equal(row_x, row_x0) and torch.equal(loss, loss0)
    scale = torch.cat((torch.full((M,), 1.0 / M), torch.full((M,), -1.0 / M))).cuda()
    d_out0, dE0 = torch.empty_like(o2), torch.zeros_like(E)
    LIB.call('acsr_bpr_loss_bwd', ops._p(o2), ops._p(E), ops._p(pos, torch.int64), ops._p(neg, torch.int64), ops._p(row_x0),
             ops._p(scale), M2, d, gamma, 0, M, ops._p(d_out0), ops._p(dE0), ops._stream())
    d_out = torch.zeros_like(o2)
    grads = []
    for (lo, hi), sh in zip(bounds, shards):
        gs = torch.zeros_like(sh)
        d_out += ops.bpr_loss_bwd_shard(o2, sh, lo, hi, V, pos, neg, row_x, scale, gamma, 0, M, gs)
        grads.append(gs)
    dE = torch.cat(grads)
    assert float((d_out - d_out0).abs().max()) <= 1e-6 * float(d_out0.abs().max())
    assert float((dE - dE0).abs().max()) <= 1e-6 * float(dE0.abs().max())
    # a rank that owns both rows of a pair computes g * (E[pos] - E[neg]) as the unsharded kernel does
    both = torch.zeros(M2, dtype=torch.bool, device='cuda')
    for lo, hi in bounds:
        both |= (pos >= lo) & (pos < hi) & (neg >= lo) & (neg < hi)
    assert torch.equal(d_out[both], d_out0[both])


def test_shard_kernel_argument_checks(A):
    ops, LIB, Err = A.ops, A.LIB, A.AcsrError
    d, M, V = 64, 4, 1000
    out = torch.randn(M, d, device='cuda')
    sh = torch.randn(100, d, device='cuda')
    cand = torch.randint(0, V, (M, 11), device='cuda')
    ids = torch.randint(0, V, (M,), device='cuda')
    sc = torch.randn(M, 11, device='cuda')
    p, s = ops._p, ops._stream()
    cases = [
        lambda: LIB.call('acsr_candidate_scores_shard', None, p(sh), 0, 100, V, d, p(cand, torch.int64), M, 11, p(sc), s),
        lambda: LIB.call('acsr_candidate_scores_shard', p(out), p(sh), 100, 100, V, d, p(cand, torch.int64), M, 11, p(sc), s),
        lambda: LIB.call('acsr_candidate_scores_shard', p(out), p(sh), 900, 1001, V, d, p(cand, torch.int64), M, 11, p(sc), s),
        lambda: LIB.call('acsr_candidate_scores_shard', p(out), p(sh), 0, 100, V, 62, p(cand, torch.int64), M, 11, p(sc), s),
        lambda: LIB.call('acsr_candidate_scores_shard', p(out), p(sh), 0, 100, V, d, p(cand, torch.int64), M, 8193, p(sc), s),
        lambda: LIB.call('acsr_candidate_scores_shard', out.data_ptr() + 4, p(sh), 0, 100, V, d, p(cand, torch.int64), M, 11, p(sc), s),
        lambda: LIB.call('acsr_candidate_scores_shard', p(out), sh.data_ptr() + 8, 0, 100, V, d, p(cand, torch.int64), M, 11, p(sc), s),
        lambda: LIB.call('acsr_candidate_rank_scores', p(sc), p(cand, torch.int64), V, M, 11, 10, None, None, s),
        lambda: LIB.call('acsr_candidate_rank_scores', p(sc), p(cand, torch.int64), V, 0, 11, 10, p(cand, torch.int64), None, s),
        lambda: LIB.call('acsr_candidate_rank_scores', p(sc), p(cand, torch.int64), V, M, 8193, 10, p(cand, torch.int64), None, s),
        lambda: LIB.call('acsr_candidate_rank_scores', p(sc), p(cand, torch.int64), V, M, 11, 1025, p(cand, torch.int64), None, s),
        lambda: LIB.call('acsr_bpr_dots_shard', p(out), p(sh), 0, 100, V, p(ids, torch.int64), None, M, d, p(sc), s),
        lambda: LIB.call('acsr_bpr_dots_shard', p(out), p(sh), 50, 10, V, p(ids, torch.int64), p(ids, torch.int64), M, d, p(sc), s),
        lambda: LIB.call('acsr_bpr_loss_from_dots', p(sc), 6, 4, 1e-10, p(sc), p(sc), p(sc), s),
        lambda: LIB.call('acsr_bpr_loss_from_dots', p(sc), M, 9, 1e-10, p(sc), p(sc), p(sc), s),
        lambda: LIB.call('acsr_bpr_loss_bwd_shard', p(out), p(sh), 0, 100, V, p(ids, torch.int64), p(ids, torch.int64), p(sc), p(sc),
                         M, d, 1e-10, 0, M, None, None, s),
        lambda: LIB.call('acsr_bpr_loss_bwd_shard', p(out), p(sh), 0, 2000, V, p(ids, torch.int64), p(ids, torch.int64), p(sc), p(sc),
                         M, d, 1e-10, 0, M, p(out), None, s),
        lambda: ops.candidate_scores_shard(out, sh, 0, 101, V, cand),
        lambda: ops.candidate_rank_scores(sc, cand[:, :5], V, 10),
    ]
    for i, c in enumerate(cases):
        with pytest.raises(Err):
            c()
        torch.cuda.synchronize()


# ---- the real VocabParallel with the CUDA kernels, gloo collectives on CPU tensors -------------------------------------------
def _vp_worker(rank, world, port, V, d, k, N, R, outdir):
    sys.path.insert(0, ROOT)
    ret = {}
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        import ac_tsr_b200 as A
        A.LIB.load()

        def cpu(r):
            return tuple(t.cpu() if t is not None else None for t in r)

        class GpuCompute(A.dist.CudaCompute):
            """the CUDA kernels on the one GPU, their results handed back on the CPU for gloo"""

            def candidate_scores_shard(self, out, shard, lo, hi, V, cand):
                return super().candidate_scores_shard(out.cuda(), shard.cuda(), lo, hi, V, cand.cuda()).cpu()

            def candidate_rank_scores(self, scores, cand, V, k, counts):
                return cpu(super().candidate_rank_scores(scores.cuda(), cand.cuda(), V, k, counts))

            def bpr_dots_shard(self, out, shard, lo, hi, V, pos, neg):
                return super().bpr_dots_shard(out.cuda(), shard.cuda(), lo, hi, V, pos.cuda(), neg.cuda()).cpu()

            def bpr_loss_from_dots(self, dots, n_groups, gamma):
                return cpu(super().bpr_loss_from_dots(dots.cuda(), n_groups, gamma))

        g = torch.Generator().manual_seed(11 * world)
        E = torch.randn(V, d, generator=g) * 0.2
        out_all = torch.randn(world, R, d, generator=g)
        vp0 = A.dist.VocabParallel(V, compute=GpuCompute(3, d))
        bounds = [(min(V, r * vp0.per), min(V, (r + 1) * vp0.per)) for r in range(world)]
        cand_all = make_cand(V, world * R, N, bounds, g).view(world, R, N + 1)
        pos_all = torch.randint(1, V, (world, 2 * R), generator=g)
        neg_all = torch.randint(1, V, (world, 2 * R), generator=g)
        out, cand = out_all[rank], cand_all[rank]
        rec0, s0, cnt0 = A.ops.candidate_rank(out.cuda(), E.cuda(), cand.cuda(), k, want_scores=True, want_counts=True)
        o2 = out.repeat(2, 1)
        loss0 = A.ops.BprLossFn.apply(o2.cuda(), E.cuda(), pos_all[rank].cuda(), neg_all[rank].cuda(), 2, 1e-10)
        for sharded in (False, True):
            key = '%d %s' % (rank, 'sharded' if sharded else 'replicated')
            try:
                vp = A.dist.VocabParallel(V, compute=GpuCompute(3, d), sharded=sharded)
                table = vp.make_shard(E) if sharded else E
                rec, sc, cnt = vp.sampled_rank(out, table, cand, k, counts=True)
                assert torch.equal(sc, s0.cpu()) and torch.equal(rec, rec0.cpu()) and torch.equal(cnt, cnt0.cpu())
                rec1, _ = vp.sampled_rank(out, table, cand, k)
                assert torch.equal(rec1, rec0.cpu())
                loss, _ = vp.bpr_forward(o2, table, pos_all[rank], neg_all[rank], 2, 1e-10)
                assert torch.equal(loss, loss0.cpu()), (loss, loss0)
                ret[key] = 'ok'
            except Exception as e:          # every rank fails alike, so the collectives of the next case still match
                ret[key] = '%s: %s' % (type(e).__name__, str(e)[:300])
    finally:
        dist.destroy_process_group()
    with open(os.path.join(outdir, 'rank%d.json' % rank), 'w') as fh:
        json.dump(ret, fh)


@pytest.mark.parametrize('W', [2, 8])
def test_vocab_parallel_sampled_rank(W, tmp_path):
    V, d, k, N, R = 60001, 64, 50, 99, 33
    port = 29450 + (os.getpid() + 5 * W) % 200
    ctx = mp.start_processes(_vp_worker, args=(W, port, V, d, k, N, R, str(tmp_path)), nprocs=W, join=False, start_method='spawn')
    deadline = time.time() + 900
    try:
        while not ctx.join(timeout=5):
            assert time.time() < deadline, 'vocab-parallel workers did not finish in time'
    finally:
        for p in ctx.processes:
            if p.is_alive():
                p.terminate()
            p.join()
    got = {}
    for r in range(W):
        with open(os.path.join(str(tmp_path), 'rank%d.json' % r)) as fh:
            got.update(json.load(fh))
    assert len(got) == W * 2
    bad = {key: v for key, v in got.items() if v != 'ok'}
    assert not bad, bad
