"""gloo tests (CPU, world size 2 and 3) of the vocab-parallel sampled ranking and BPR loss (ac-tsr_b200/dist.py): with torch
restatements of the five local kernels injected, VocabParallel.sampled_rank must rank exactly as the unsharded candidate
ranking, and bpr_forward / bpr_backward must give the unsharded BPR loss, d_out and table gradient, for both storage modes."""
import os
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _rows(shard, ids, lo, hi):
    """shard rows of the ids, 0 for ids this rank does not own"""
    own = (ids >= lo) & (ids < hi)
    return shard[(ids - lo).clamp(0, shard.shape[0] - 1)] * own.to(shard.dtype).unsqueeze(-1), own


def rank_rows(scores, cand, V, k):
    """acsr_candidate_rank's ranking: distinct negatives above / tied with the positive, distinct candidates"""
    ids = cand.clamp(0, V - 1)
    M = scores.shape[0]
    counts = torch.zeros((M, 3), dtype=torch.int32)
    for m in range(M):
        seen, s0 = {int(ids[m, 0])}, float(scores[m, 0])
        for c in range(1, ids.shape[1]):
            i = int(ids[m, c])
            if i in seen:
                continue
            seen.add(i)
            counts[m, 0] += int(float(scores[m, c]) > s0)
            counts[m, 1] += int(float(scores[m, c]) == s0)
        counts[m, 2] = len(seen)
    rec = torch.zeros((M, k + 1), dtype=torch.int32)
    rec[:, k] = 1
    hit = counts[:, 0] < k
    rec[hit.nonzero().view(-1), counts[hit, 0].long()] = 1
    return rec, counts


class TorchCompute(object):
    def candidate_scores_shard(self, out, shard, lo, hi, V, cand):
        rows, _ = _rows(shard, cand.clamp(0, V - 1), lo, hi)                 # [M, C, d]
        return (out.unsqueeze(1) * rows).sum(-1)

    def candidate_rank_scores(self, scores, cand, V, k, counts):
        rec, cnt = rank_rows(scores, cand, V, k)
        return rec, (cnt if counts else None)

    def bpr_dots_shard(self, out, shard, lo, hi, V, pos, neg):
        ep, _ = _rows(shard, pos, lo, hi)
        en, _ = _rows(shard, neg, lo, hi)
        return torch.stack(((out * ep).sum(1), (out * en).sum(1)), 1)

    def bpr_loss_from_dots(self, dots, n_groups, gamma):
        x = dots[:, 0] - dots[:, 1]
        return (-torch.log(gamma + torch.sigmoid(x))).view(n_groups, -1).mean(1), x

    def bpr_loss_bwd_shard(self, out, shard, lo, hi, V, pos, neg, row_x, row_scale, gamma, row_begin, row_end, shard_grad):
        s = torch.sigmoid(row_x)
        g = -row_scale * s * (1 - s) / (gamma + s)
        ep, op = _rows(shard, pos, lo, hi)
        en, on = _rows(shard, neg, lo, hi)
        if shard_grad is not None:
            sl = slice(row_begin, row_end)
            v = g[sl, None] * out[sl]
            shard_grad.index_add_(0, (pos[sl] - lo)[op[sl]], v[op[sl]])
            shard_grad.index_add_(0, (neg[sl] - lo)[on[sl]], -v[on[sl]])
        return g[:, None] * (ep - en)


def boundary_ids(vp):
    """0, the last item, every shard's first and last row and the rows next to them, and two out-of-range ids"""
    ids = {0, vp.V - 1, -3, vp.V + 5}
    for r in range(vp.world):
        lo = min(vp.V, r * vp.per)
        hi = min(vp.V, lo + vp.per)
        ids.update(i for i in (lo - 1, lo, hi - 1, hi) if 0 <= i < vp.V)
    return sorted(ids)


def _worker(rank, world, port, V, ret):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        import ac_tsr_b200 as A
        g = torch.Generator().manual_seed(V + world)
        d, R, N, k, gamma = 8, 12, 14, 5, 1e-10
        # small integer embeddings: many exact ties between candidates
        E = torch.randint(-2, 3, (V, d), generator=g).double()
        out_all = torch.randint(-2, 3, (world, R, d), generator=g).double()
        out_all[:, 3] = 0                                                   # every candidate ties with the positive
        vp0 = A.dist.VocabParallel(V, compute=TorchCompute(), align=8)
        assert vp0.shard_rows[-1] < vp0.per                                 # the last shard is the small one
        edge = torch.tensor(boundary_ids(vp0))
        cand_all = torch.randint(1, V, (world, R, 1 + N), generator=g)
        cand_all[:, :, 1:1 + edge.numel()] = edge                           # boundary, id 0 and out-of-range ids
        cand_all[:, ::3, 0] = edge[torch.arange(cand_all[:, ::3, 0].numel()) % edge.numel()].view(world, -1)
        cand_all[:, :, -3:-1] = cand_all[:, :, -4:-3]                       # duplicates
        cand_all[:, ::2, -1] = cand_all[:, ::2, 0]                          # the positive again among the negatives
        out, cand = out_all[rank].clone(), cand_all[rank].clone()
        # unsharded references
        ids = cand.clamp(0, V - 1)
        s_ref = (out.unsqueeze(1) * E[ids]).sum(-1)
        rec_ref, cnt_ref = rank_rows(s_ref, cand, V, k)
        assert int(cnt_ref[:, 1].max()) > 0 and int((cnt_ref[:, 2] < N + 1).sum()) > 0
        pos_all = torch.randint(1, V, (world, 2 * R), generator=g)
        neg_all = torch.randint(0, V, (world, 2 * R), generator=g)
        pos_all[:, :edge.numel() - 2] = edge[1:-1]
        neg_all[:, 1:edge.numel() - 1] = edge[1:-1]                         # pos / neg on different shards, and on the same
        neg_all[:, ::5] = pos_all[:, ::5]
        pos_all[pos_all < 0] = 0
        pos_all[pos_all >= V] = V - 1
        neg_all[neg_all < 0] = 0
        neg_all[neg_all >= V] = V - 1
        pos, neg = pos_all[rank].clone(), neg_all[rank].clone()
        scale = torch.cat((torch.full((R,), 1.0 / R, dtype=torch.float64), torch.full((R,), -1.0 / R, dtype=torch.float64)))
        o = out_all.repeat(1, 2, 1)[rank].clone().requires_grad_(True)       # [calibrated ; attacked] rows
        Eg = E.clone().requires_grad_(True)
        x = (o * Eg[pos]).sum(1) - (o * Eg[neg]).sum(1)
        rl = -torch.log(gamma + torch.sigmoid(x))
        loss_ref = rl.view(2, R).mean(1)
        (rl * scale).sum().backward(inputs=[o])
        tot = 0                                                             # the calibrated rows of every rank train the table
        for r in range(world):
            orr = out_all[r]
            xr = (orr * Eg[pos_all[r, :R]]).sum(1) - (orr * Eg[neg_all[r, :R]]).sum(1)
            tot = tot + (-torch.log(gamma + torch.sigmoid(xr)) / R).sum()
        tot.backward(inputs=[Eg])
        for sharded in (False, True):
            vp = A.dist.VocabParallel(V, compute=TorchCompute(), align=8, sharded=sharded)
            table = vp.make_shard(E) if sharded else E
            rec, scores, cnt = vp.sampled_rank(out, table, cand, k, counts=True)
            assert torch.equal(scores, s_ref), sharded
            assert torch.equal(rec, rec_ref) and torch.equal(cnt, cnt_ref), sharded
            rec2, _ = vp.sampled_rank(out, table, cand, k)
            assert torch.equal(rec2, rec_ref)
            loss, st = vp.bpr_forward(o.detach(), table, pos, neg, 2, gamma)
            assert torch.allclose(loss, loss_ref, rtol=1e-12, atol=0), (sharded, loss, loss_ref)
            tg = torch.zeros_like(table)
            d_out = vp.bpr_backward(st, table, scale, tg, table_half=0)
            assert torch.allclose(d_out, o.grad, rtol=0, atol=1e-12), sharded
            assert torch.allclose(vp.shard(tg), Eg.grad[vp.lo:vp.hi], rtol=0, atol=1e-12), sharded
            rest = torch.ones(tg.shape[0], dtype=torch.bool)
            rest[(0 if sharded else vp.lo):(vp.hi - vp.lo if sharded else vp.hi)] = False
            assert not bool(tg[rest].any()), sharded                                 # nothing outside the owned rows
        ret[rank] = 'ok'
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize('world,V', [(2, 37), (2, 90), (3, 50), (3, 61)])
def test_vocab_parallel_sampled_rank_and_bpr(world, V):
    mgr = mp.Manager()
    ret = mgr.dict()
    port = 29300 + (os.getpid() + 7 * V + world) % 250
    mp.spawn(_worker, args=(world, port, V, ret), nprocs=world, join=True)
    assert dict(ret) == {r: 'ok' for r in range(world)}
