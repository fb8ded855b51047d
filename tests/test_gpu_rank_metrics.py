"""Rank counts of the positive (GAUC) on every full-sort path and in sampled ranking, and GAUC / the item-distribution metrics
end to end.

The exact tests reuse the integer cases of test_gpu_topk.py: every score is an integer the kernels compute exactly, so the counts
G = #items above the positive and E = #items tied with it (column 0 and the positive itself left out) must equal a float64
reference with no tolerance, on rows designed around ties (constant rows: the positive ties with every item)."""
import json
import os
import sys
import time

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
import test_gpu_topk as T                                     # noqa: E402  (make_case / reference)
from oracle import metrics_oracle as MO                       # noqa: E402
from oracle import acsr_oracle as O                           # noqa: E402

GOLD = os.path.join(ROOT, 'tests', 'golden')


@pytest.fixture(scope='module')
def A():
    import ac_tsr_b200 as pkg
    pkg.LIB.load()
    return pkg


def ref_scores(out, E, skip_col0=True):
    s = out.double() @ E.double().t()
    if skip_col0:
        s[:, 0] = -float('inf')
    return s


def positives(s, seed):
    """per row in turn: the best item, the worst item (column 0 aside), a random item"""
    g = torch.Generator().manual_seed(seed)
    s = s.cpu()
    best = s.argmax(1)
    t = s.clone()
    t[:, 0] = float('inf')
    worst = t.argmin(1)
    rnd = torch.randint(1, s.shape[1], (s.shape[0],), generator=g)
    r = torch.arange(s.shape[0]) % 3
    return torch.where(r == 0, best, torch.where(r == 1, worst, rnd))


def ref_counts(s, pos):
    """float64 (G, E) with the positive's own column excluded"""
    sp = s.gather(1, pos.view(-1, 1).to(s.device))
    gt = (s > sp).sum(1)
    eq = (s == sp).sum(1) - 1
    return torch.stack((gt, eq), 1).cpu()


def check(A, out, E, k, seed, what, **kw):
    s = ref_scores(out, E)
    pos = positives(s, seed).cuda()
    want = ref_counts(s, pos)
    val, idx, rec, counts = A.ops.full_sort_topk(out, E, k, pos, counts=True, **kw)
    assert counts.dtype == torch.int32 and tuple(counts.shape) == (out.shape[0], 2)
    bad = (counts.cpu().long() != want).any(1).nonzero().view(-1)
    assert bad.numel() == 0, (what, bad[:8].tolist(), counts[bad[:4]].tolist(), want[bad[:4]].tolist())
    v0, i0, r0 = A.ops.full_sort_topk(out, E, k, pos, **kw)
    assert torch.equal(val, v0), what                           # counting leaves the top-k values untouched
    return want, (val, idx, rec), (v0, i0, r0)


@pytest.mark.parametrize('V,d', [(5000, 64), (5001, 32), (50000, 128)])
def test_select_path_counts_exact(A, V, d):
    out, E, _ = T.make_case(V, d, 10, 130, seed=V + d)
    want, _, _ = check(A, out, E, 10, 1, 'select V=%d d=%d' % (V, d))
    assert int(want[:, 1].max()) >= V - 3                       # a constant row: the positive ties with every other item


@pytest.mark.parametrize('M', [1, 130, 256])
@pytest.mark.parametrize('k', [10, 64])
def test_fused_tcgen05_counts_exact(A, M, k):
    V = 100003                                                  # above the select limit, ragged last tile and chunk
    out, E, _ = T.make_case(V, 64, k, M, seed=M + k)
    for share in (True, False):
        s = ref_scores(out, E)
        pos = positives(s, 3).cuda()
        want = ref_counts(s, pos)
        sp = A.ops.row_dot(out, E, pos)
        pv, pi, pc = A.ops.logits_topk_rank_partial(out, E, k, pos, sp, share_bound=share)
        val, idx, rec, counts = A.ops.topk_merge_rank(pv, pi, k, pc, pos)
        assert torch.equal(counts.cpu().long(), want), (M, k, share)
        pv0, pi0 = A.ops.logits_topk_partial(out, E, k, share_bound=share)
        v0, i0, r0 = A.ops.topk_merge(pv0, pi0, k, pos)
        assert torch.equal(val, v0)


@pytest.mark.parametrize('d', [32, 128])
def test_simt_counts_exact(A, d):
    out, E, _ = T.make_case(60001, d, 50, 130, seed=d)
    check(A, out, E, 50, 2, 'simt d=%d' % d)


def test_gaussian_counts_and_bitwise_topk(A):
    """Gaussian scores: the counts agree with the stored tensor-core scores except for items within 2e-6 max|score| of s_pos, and
    the top-k values, ids and hit flags are bitwise those of the top-k without counting"""
    g = torch.Generator(device='cuda').manual_seed(5)
    for V in (12102, 1000001):
        M = 256
        out = torch.randn(M, 64, generator=g, device='cuda')
        E = torch.randn(V, 64, generator=g, device='cuda') * 0.1
        pos = torch.randint(1, V, (M,), generator=g, device='cuda')
        pos[:3] = ref_scores(out[:3], E).argmax(1)
        val, idx, rec, counts = A.ops.full_sort_topk(out, E, 50, pos, counts=True)
        v0, i0, r0 = A.ops.full_sort_topk(out, E, 50, pos)
        assert torch.equal(val, v0) and torch.equal(idx, i0) and torch.equal(rec, r0), V
        sc = A.ops.logits_scores(out, E).double()
        sc[:, 0] = -float('inf')
        sp = A.ops.row_dot(out, E, pos).double().view(-1, 1)
        tol = 2e-6 * float(sc[:, 1:].abs().max())
        own = torch.zeros_like(sc, dtype=torch.bool).scatter_(1, pos.view(-1, 1), True)
        lo = ((sc > sp + tol) & ~own).sum(1)
        hi = ((sc >= sp - tol) & ~own).sum(1)
        c = counts.long()
        assert bool((c[:, 0] >= lo).all()) and bool((c[:, 0] + c[:, 1] <= hi).all()), V


def test_candidate_rank_counts(A):
    """duplicates among the negatives (and of the positive), ties: distinct counts"""
    g = torch.Generator().manual_seed(4)
    V, d, M, N = 500, 64, 300, 120
    E = torch.randint(-2, 3, (V, d), generator=g).float()
    E[:, 0] = 0
    out = torch.randint(-2, 3, (M, d), generator=g).float()
    cand = torch.randint(1, V, (M, N + 1), generator=g)
    cand[:, 5:15] = cand[:, 1:2]                                   # duplicates
    cand[::4, 20] = cand[::4, 0]                                   # the positive again among the negatives
    out[::5] = 0                                                   # every candidate ties with the positive
    rec, _, counts = A.ops.candidate_rank(out.cuda(), E.cuda(), cand.cuda(), 50, want_counts=True)
    rec0, _ = A.ops.candidate_rank(out.cuda(), E.cuda(), cand.cuda(), 50)
    assert torch.equal(rec, rec0)
    s = (out.double() @ E.double().t())
    for m in range(M):
        p = int(cand[m, 0])
        negs = sorted(set(cand[m, 1:].tolist()) - {p})
        sn = s[m, negs]
        want = [int((sn > s[m, p]).sum()), int((sn == s[m, p]).sum()), len(negs) + 1]
        assert counts[m].tolist() == want, (m, counts[m].tolist(), want)


# ---- vocab-parallel: the real VocabParallel with the CUDA kernels, gloo collectives on CPU tensors -----------------------
def _vp_worker(rank, world, port, V, d, k, Rs, outdir):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, HERE)
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

            def topk_partial(self, out, table, k, idx_offset, skip_col0):
                return cpu(super().topk_partial(out.cuda(), table.cuda(), k, idx_offset, skip_col0))

            def topk_merge(self, pv, pi, k, positive):
                return cpu(super().topk_merge(pv.cuda(), pi.cuda(), k, positive.cuda() if positive is not None else None))

            def row_dot(self, out, table, ids, idx_offset):
                return super().row_dot(out.cuda(), table.cuda(), ids.cuda(), idx_offset).cpu()

            def topk_rank_partial(self, out, table, k, positive, pos_score, idx_offset, skip_col0):
                return cpu(super().topk_rank_partial(out.cuda(), table.cuda(), k, positive.cuda(), pos_score.cuda(), idx_offset, skip_col0))

            def topk_merge_rank(self, pv, pi, k, pc, positive):
                return cpu(super().topk_merge_rank(pv.cuda(), pi.cuda(), k, pc.cuda(), positive.cuda() if positive is not None else None))

        for R in Rs:
            seed = 13 * R + world
            out_all, E, _ = T.make_case(V, d, k, world * R, seed)
            mine = slice(rank * R, (rank + 1) * R)
            out = out_all[mine]
            s = ref_scores(out, E)
            pos = positives(s, seed)
            want = ref_counts(s, pos)
            for sharded in (False, True):
                key = '%d R=%d %s' % (rank, R, 'sharded' if sharded else 'replicated')
                try:
                    vp = A.dist.VocabParallel(V, compute=GpuCompute(3, d), sharded=sharded)
                    table = vp.make_shard(E) if sharded else E
                    val, idx, rec, counts = vp.full_sort_topk(out.cpu(), table.cpu(), k, pos, counts=True)
                    assert torch.equal(counts.long(), want), (counts[:4].tolist(), want[:4].tolist())
                    v0, _, _ = vp.full_sort_topk(out.cpu(), table.cpu(), k, pos)
                    assert torch.equal(val, v0)
                    ret[key] = 'ok'
                except Exception as e:          # every rank fails alike, so the collectives of the next case still match
                    ret[key] = '%s: %s' % (type(e).__name__, str(e)[:300])
    finally:
        dist.destroy_process_group()
    with open(os.path.join(outdir, 'rank%d.json' % rank), 'w') as fh:
        json.dump(ret, fh)


@pytest.mark.parametrize('W', [2, 8])
def test_vocab_parallel_counts(W, tmp_path):
    V, d, k, Rs = 60001, 64, 10, (1, 17)
    port = 29700 + (os.getpid() + 7 * W) % 250
    ctx = mp.start_processes(_vp_worker, args=(W, port, V, d, k, Rs, str(tmp_path)), nprocs=W, join=False, start_method='spawn')
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
    assert len(got) == W * len(Rs) * 2
    bad = {key: v for key, v in got.items() if v != 'ok'}
    assert not bad, bad


# ---- end to end on ml-100k ---------------------------------------------------------------------------------------------
NEW = ['GAUC', 'ItemCoverage', 'AveragePopularity', 'GiniIndex', 'ShannonEntropy', 'TailPercentage']


def ml100k_config(A, name, mode='full', **extra):
    cd = dict(data_path=GOLD + '/', load_col={'inter': ['user_id', 'item_id', 'rating', 'timestamp']},
              eval_args={'split': {'LS': 'valid_and_test'}, 'group_by': 'user', 'order': 'TO', 'mode': mode},
              device=torch.device('cuda'), train_batch_size=256, eval_batch_size=256, seed=42, loss_type='CE', epochs=1,
              topk=[1, 10, 50], metrics=['Hit', 'GAUC', 'MRR'] + (NEW[1:] if mode == 'full' else []) + ['NDCG'],
              valid_metric='GAUC', tail_ratio=0.5, checkpoint_dir='/tmp/acsr_ckpt_rank')
    cd.update(O.default_cfg())
    cd.update(time_span=64, user_hidden_size=32, item_hidden_size=32, mask_ratio=0.2)
    if name == 'AcBERT4Rec':
        cd.update(combine_option='fixed')         # combine_option 'gate' cannot run on L + 1 positions (config/ml-100k-acbert4rec.yaml)
    cd.update(extra)
    return A.Config(model=name, dataset='ml-100k', config_dict=cd)


@pytest.mark.parametrize('name', ['ACSASRec', 'AcBERT4Rec', 'ACSSEPT', 'ACTiSASRec'])
def test_trainer_evaluate_new_metrics_ml100k(A, name, tmp_path):
    config = ml100k_config(A, name, checkpoint_dir=str(tmp_path))
    tr, va, te = A.data_preparation(config, A.create_dataset(config))
    torch.manual_seed(0)
    model = getattr(A, name)(config, tr.dataset).cuda()
    trainer = getattr(A, name + 'Trainer')(config, model)
    trainer._train_epoch(tr, 0)
    trainer.set_item_counts(tr)
    res_g = trainer.evaluate(te, load_best_model=False)                    # graphed
    trainer.use_graph = False
    res_e = trainer.evaluate(te, load_best_model=False)                    # eager
    assert res_g == res_e
    assert list(res_g)[:4] == ['hit@1', 'hit@10', 'hit@50', 'gauc']
    trainer.fused_topk = False
    res_m = trainer.evaluate(te, load_best_model=False)                    # materialised scores + torch.topk
    # the oracle on the materialised scores (the reference's full_sort_predict route)
    model.eval()
    scores, positive = [], []
    with torch.no_grad():
        for inter, _, _, pos in te:
            r = model.full_sort_predict(inter.to('cuda'))
            sc = r[1] if isinstance(r, tuple) else r
            sc = sc.view(-1, te.dataset.item_num).float().cpu()
            sc[:, 0] = -float('inf')
            scores.append(sc)
            positive.append(pos.cpu())
    scores, positive = torch.cat(scores), torch.cat(positive)
    items = torch.topk(scores, 50, dim=1)[1].numpy()
    counter = {int(i): int(n) for i, n in enumerate(trainer.item_counts) if n > 0}
    want = MO.evaluate([m.lower() for m in NEW], [1, 10, 50], scores, positive, items, te.dataset.item_num, counter, 0.5)
    for key, v in want.items():
        assert abs(res_g[key] - v) <= 2e-3, (name, key, res_g[key], v)              # modulo near-ties between the paths
        assert abs(res_m[key] - v) <= 1e-4, (name, key, res_m[key], v)

    # sampled evaluation (uni100): GAUC next to the top-k metrics, graphed == eager
    cs = ml100k_config(A, name, mode='uni100', checkpoint_dir=str(tmp_path))
    _, _, te_s = A.data_preparation(cs, A.create_dataset(cs))
    ts = getattr(A, name + 'Trainer')(cs, model)
    s = te_s.neg_sampler
    s.to_device('cuda')
    st = s.rng.state.clone()
    rs_g = ts.evaluate(te_s, load_best_model=False)
    s.rng.state.copy_(st)
    ts.use_graph = False
    rs_e = ts.evaluate(te_s, load_best_model=False)
    assert rs_g == rs_e and 0.0 <= rs_g['gauc'] <= 1.0
    cs_bad = ml100k_config(A, name, mode='uni100', metrics=['Recall', 'ItemCoverage'], checkpoint_dir=str(tmp_path))
    with pytest.raises(NotImplementedError, match='sampled evaluation'):
        getattr(A, name + 'Trainer')(cs_bad, model).evaluate(te_s, load_best_model=False)


def test_run_recbole_with_the_new_metrics(A, tmp_path):
    import subprocess
    cfg = tmp_path / 'rank.yaml'
    cfg.write_text('metrics: [Recall, GAUC, ItemCoverage, AveragePopularity, GiniIndex, ShannonEntropy, TailPercentage, NDCG]\n'
                   'topk: [10]\nvalid_metric: GAUC\nepochs: 1\ncheckpoint_dir: %s\n' % tmp_path)
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'run_recbole.py'), '--config_files',
                        os.path.join(ROOT, 'config', 'ml-100k.yaml') + ' ' + str(cfg)],
                       cwd=ROOT, capture_output=True, text=True, timeout=900)
    log = r.stdout + r.stderr
    assert r.returncode == 0, log[-3000:]
    assert 'gauc' in log and 'giniindex@10' in log and 'tailpercentage@10' in log, log[-3000:]
