"""Negative sampling on the device (acsr_neg_sample) and sampled-candidate ranking (acsr_candidate_rank) on the B200: sampler
properties, the ranking against the oracle's RecBole-style scatter + topk, sampled evaluation through the trainer for the four
models, training RNG isolation, BPR training with sampled negatives, and run_recbole end to end.  The reference cannot run
here, so no golden comes from it: every check is against the oracle's plain restatement of RecBole's semantics."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import acsr_oracle as O
from oracle import negsample_oracle as NO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, 'tests', 'golden')


@pytest.fixture(scope='module')
def A():
    import ac_tsr_b200 as pkg
    pkg.LIB.load()
    return pkg


def make_config(A, cfg, model='ACSASRec', **extra):
    d = dict(cfg)
    d.update(USER_ID_FIELD='user_id', ITEM_ID_FIELD='item_id', LIST_SUFFIX='_list', ITEM_LIST_LENGTH_FIELD='item_length',
             NEG_PREFIX='neg_', TIME_FIELD='timestamp', device=torch.device('cuda'), seed=42, learning_rate=1e-3, epochs=1,
             eval_batch_size=256, train_batch_size=256, topk=[1, 5, 10, 50], metrics=['Hit', 'MRR', 'NDCG', 'Recall'],
             valid_metric='Hit@10', checkpoint_dir='/tmp/acsr_ckpt_neg', cuda_graph=True)
    d.update(extra)
    return A.Config(model=model, config_dict=d)


def ml100k_config(A, **extra):
    cd = dict(data_path=GOLD + '/', load_col={'inter': ['user_id', 'item_id', 'rating', 'timestamp']},
              eval_args={'split': {'LS': 'valid_and_test'}, 'group_by': 'user', 'order': 'TO', 'mode': 'full'},
              device=torch.device('cuda'), train_batch_size=256, eval_batch_size=256, seed=42, loss_type='CE', epochs=1,
              topk=[1, 5, 10, 50], metrics=['Hit', 'MRR', 'NDCG', 'Recall'], valid_metric='Hit@10', checkpoint_dir='/tmp/acsr_ckpt_neg')
    cd.update(O.default_cfg())
    cd.update(extra)
    return A.Config(model='ACSASRec', dataset='ml-100k', config_dict=cd)


@pytest.fixture(scope='module')
def ml100k(A):
    config = ml100k_config(A)
    ds = A.create_dataset(config)
    return config, ds, ds.build()


def draw_many(s, users, N, positives=None, reps=1):
    out = []
    for _ in range(reps):
        out.append(s.draw(users, N, positives=positives).cpu())
    return torch.cat(out)


def check_excluded(negs, users, off, items, n_items):
    negs, users = negs.numpy(), users.cpu().numpy()
    assert negs.min() >= 1 and negs.max() < n_items
    for r in range(negs.shape[0]):
        u = users[r]
        used = items[off[u]:off[u + 1]]
        assert not np.isin(negs[r], used).any(), r


# ---- sampler properties ----------------------------------------------------------------------------------------
@pytest.mark.parametrize('dist', ['uniform', 'popularity'])
def test_sampler_properties_ml100k(A, ml100k, dist):
    from scipy.stats import chisquare
    config, ds, splits = ml100k
    s = A.dataset.build_neg_samplers(config, splits, None, dist)[2]            # test phase: the largest used sets
    te = splits[2].inter_feat
    users, pos = te['user_id'].cuda(), te['item_id'].cuda()
    negs = s.draw(users, 100, positives=pos).cpu()
    check_excluded(negs, users, s.used_offsets, s.used_items, ds.item_num)
    # one user, many draws: frequencies over the complement against the exact distribution
    # a user of median history (for popularity, a heavy user's used set can hold enough of the mass that the bounded alias
    # retries give way to the uniform-complement draw now and then, which this exact-distribution test would flag)
    sizes = np.diff(s.used_offsets)
    u = int(np.argsort(sizes)[len(sizes) // 2])
    used = set(s.used_items[s.used_offsets[u]:s.used_offsets[u + 1]].tolist())
    comp = np.array([i for i in range(1, ds.item_num) if i not in used])
    many = draw_many(s, torch.full((512,), u, dtype=torch.int64, device='cuda'), 256, reps=4).reshape(-1).numpy()
    assert not np.isin(many, list(used)).any()
    cnt = np.bincount(many, minlength=ds.item_num)[comp].astype(np.float64)
    if dist == 'uniform':
        p = np.full(len(comp), 1.0 / len(comp))
    else:
        p = s.counts[comp] / s.counts[comp].sum()
    keep = p * many.size >= 5                                                 # chi-square cells with enough expected mass
    exp = p[keep] * many.size
    obs = cnt[keep]
    exp *= obs.sum() / exp.sum()
    assert chisquare(obs, exp).pvalue > 1e-4
    if dist == 'popularity':                                                  # items that never were a target are never drawn
        assert cnt[s.counts[comp] == 0].sum() == 0


def test_sampler_properties_million_items(A):
    from scipy.stats import chisquare
    V, U = 1_000_001, 257
    rng = np.random.default_rng(3)
    uid = np.repeat(np.arange(1, U), 400)
    iid = rng.integers(1, V, size=uid.size)
    off, items = A.ops.used_item_csr(uid, iid, U, V)
    s = A.ops.NegSampler('uniform', off, items, V, seed=5)
    users = torch.arange(1, U, dtype=torch.int64, device='cuda')
    negs = s.draw(users, 1000).cpu()
    check_excluded(negs, users, off, items, V)
    # uniform over the complement: ranks of the draws among the complement items, in 100 equal bins
    u = 7
    used = items[off[u]:off[u + 1]]
    many = draw_many(s, torch.full((1024,), u, dtype=torch.int64, device='cuda'), 512, reps=2).reshape(-1).numpy()
    assert not np.isin(many, used).any()
    rank = many - 1 - np.searchsorted(used, many)                           # position in the complement
    n_comp = V - 1 - len(used)
    obs = np.bincount(rank * 100 // n_comp, minlength=100)
    assert chisquare(obs).pvalue > 1e-4
    # popularity over a Zipf catalogue, with the used sets excluded
    counts = np.zeros(V)
    counts[1:] = 1.0 / np.arange(1, V)
    sp = A.ops.NegSampler('popularity', off, items, V, seed=5, counts=counts)
    negs = sp.draw(users, 1000).cpu()
    check_excluded(negs, users, off, items, V)
    top = np.bincount(negs.reshape(-1).numpy(), minlength=V)[1:11].astype(np.float64)
    # expected share of item i: sum over users of p_u(i) -- computed for the 10 most popular items
    exp = np.zeros(10)
    for uu in range(1, U):
        ex = np.zeros(V, dtype=bool)
        ex[items[off[uu]:off[uu + 1]]] = True
        w = counts * (~ex)
        exp += 1000 * w[1:11] / w.sum()
    assert np.all(np.abs(top - exp) < 6 * np.sqrt(exp) + 5)


def test_sampler_determinism_and_single_item_complement(A):
    V = 50
    uid = np.array([1] * (V - 2) + [2, 2])
    iid = np.concatenate([np.arange(1, V - 1), [3, 4]])                   # user 1: only item V-1 is left
    off, items = A.ops.used_item_csr(uid, iid, 3, V)
    for dist in ('uniform', 'popularity'):
        s = A.ops.NegSampler(dist, off, items, V, seed=11, counts=np.r_[0.0, np.ones(V - 1)])
        users = torch.tensor([1, 2, 0, 1], dtype=torch.int64, device='cuda')
        s.to_device('cuda')
        st = s.rng.state.clone()
        a = s.draw(users, 64).cpu()
        b = s.draw(users, 64).cpu()
        s.rng.state.copy_(st)
        a2 = s.draw(users, 64).cpu()
        assert torch.equal(a, a2) and not torch.equal(a, b)
        assert (a[0] == V - 1).all() and (a[3] == V - 1).all() and (b[0] == V - 1).all()
        assert not np.isin(a[1].numpy(), [3, 4]).any() and a.min() >= 1
        # the positive is excluded too when it lies outside the used set
        c = s.draw(torch.tensor([2], device='cuda'), 256, positives=torch.tensor([7], device='cuda')).cpu()
        assert not np.isin(c.numpy(), [3, 4, 7]).any()


# ---- acsr_candidate_rank against the oracle -----------------------------------------------------------------------
@pytest.mark.parametrize('d', [32, 64, 128, 256])
@pytest.mark.parametrize('N', [1, 99, 1000])
def test_candidate_rank_vs_oracle(A, d, N):
    g = torch.Generator().manual_seed(d * 7 + N)
    B, V, kmax = 64, 5000, 50
    out = torch.randn(B, d, generator=g) * 0.3
    table = torch.randn(V, d, generator=g) * 0.3
    cand = torch.randint(1, V, (B, 1 + N), generator=g)
    if N > 1:
        cand[:, 2] = cand[:, 1]                                              # forced duplicates
        cand[::3, 1 + N // 2] = cand[::3, 1]
        # forced exact ties: a negative whose table row equals the positive's
        table[V - 1] = table[cand[5, 0]]
        cand[5, N] = V - 1
    out_c, table_c, cand_c = out.cuda(), table.cuda(), cand.cuda()
    rec, scores = A.ops.candidate_rank(out_c, table_c, cand_c, kmax, want_scores=True)
    ref_scores = (out.double().unsqueeze(1) * table.double()[cand]).sum(-1)
    assert float((scores.cpu().double() - ref_scores).abs().max()) <= 1e-5 * float(ref_scores.abs().max())
    rec = rec.cpu()
    assert torch.equal(rec[:, kmax], torch.ones(B, dtype=torch.int32)) and (rec[:, :kmax].sum(1) <= 1).all()
    flags, _, full = NO.sampled_topk(ref_scores, cand, V, kmax)
    lo, hi = NO.sampled_rank_bounds(full, cand[:, 0], tol=2e-6 * float(ref_scores.abs().max()))
    r_gpu, r_or = NO.flags_rank(rec, kmax), NO.flags_rank(flags, kmax)
    ok = lambda r: ((r >= lo.clamp(max=kmax)) & (r <= hi.clamp(max=kmax))).all()       # noqa: E731
    assert bool(ok(r_gpu)) and bool(ok(r_or))
    same = lo == hi
    assert torch.equal(r_gpu[same], r_or[same])
    if N > 1:
        assert int(r_gpu[5]) == min(int(lo[5]), kmax)                      # an exact tie counts for the positive


def test_candidate_rank_rejects_beyond_limit(A):
    out, table = torch.zeros(2, 64, device='cuda'), torch.zeros(10, 64, device='cuda')
    with pytest.raises(A.AcsrError, match='8191'):
        A.ops.candidate_rank(out, table, torch.ones(2, 8193, dtype=torch.int64, device='cuda'), 10)


# ---- trained-model invariant and trainer.evaluate -------------------------------------------------------------------
def test_sampled_rank_never_worse_than_full_sort_rank(A, ml100k, tmp_path):
    config, ds, splits = ml100k
    config = ml100k_config(A, checkpoint_dir=str(tmp_path))
    tr, va, te = A.data_preparation(config, A.create_dataset(config))
    model = A.ACSASRec(config, tr.dataset).cuda()
    trainer = A.ACSASRecTrainer(config, model)
    trainer._train_epoch(tr, 0)
    model.eval()
    s = A.dataset.build_neg_samplers(config, splits, None, 'uniform')[2]
    kmax = 50
    inter = te.dataset.inter_feat.to('cuda')
    pos = inter['item_id']
    cand = torch.empty((len(pos), 101), dtype=torch.int64, device='cuda')
    s.draw(inter['user_id'], 100, positives=pos, out=cand[:, 1:], ld=101)
    with torch.no_grad():
        sc, rec_s = model.sampled_topk(inter, cand, kmax, pos)
        _, full = model.full_sort_predict(inter)
    full = full.double().cpu()
    full[:, 0] = -float('inf')
    s0 = full.gather(1, pos.cpu().view(-1, 1))
    tol = 2e-6 * float(full[:, 1:].abs().max())
    # the full-sort rank up to ties between the two paths' scores (3xTF32 tensor cores vs fp32 FMA): at most the number of
    # items scoring at least s_pos - tol
    full_rank_hi = (full >= s0 - tol).sum(1) - 1
    r_s = NO.flags_rank(rec_s.cpu(), kmax)
    assert bool((r_s <= full_rank_hi.clamp(max=kmax)).all())
    for k in (1, 10, 50):                                                  # per row: a full-sort hit is a sampled hit
        assert bool(((r_s < k) | (full_rank_hi >= k)).all())


def _synthetic_c2(A, name, mode):
    """C2 shape (V = 12 102, the default encoder: 2 layers, 2 heads, d 64, inner 256), 512 evaluation users"""
    cfg = O.default_cfg()
    cfg.update(time_span=64, user_hidden_size=32, item_hidden_size=32, mask_ratio=0.2)
    extra = dict(MAX_ITEM_LIST_LENGTH=49) if name == 'AcBERT4Rec' else {}
    config = make_config(A, cfg, model=name, **extra)
    V, n = 12102, 512
    ds = A.data.SyntheticSequentialDataset(config, n, V, seed=9)
    f = ds.inter_feat
    uid, iid = f['user_id'].numpy(), f['item_id'].numpy()
    off, items = A.ops.used_item_csr(uid, iid, n + 1, V)
    counts = np.bincount(iid, minlength=V).astype(np.float64)
    s = A.ops.NegSampler(mode, off, items, V, seed=42, phase=1, counts=counts)
    loader = A.data.NegSampleEvalDataLoader(config, ds, s, 100)
    torch.manual_seed(1)
    model = getattr(A, name)(config, ds).cuda()
    trainer = getattr(A, name + 'Trainer')(config, model)
    return config, ds, loader, model, trainer


@pytest.mark.parametrize('mode', ['uniform', 'popularity'])
@pytest.mark.parametrize('name', ['ACSASRec', 'AcBERT4Rec', 'ACSSEPT', 'ACTiSASRec'])
def test_trainer_sampled_evaluate_matches_oracle(A, name, mode):
    config, ds, loader, model, trainer = _synthetic_c2(A, name, mode)
    s = loader.neg_sampler
    s.to_device('cuda')
    st = s.rng.state.clone()
    result = trainer.evaluate(loader, load_best_model=False)                # graphed sampled evaluation
    assert all(np.isfinite(v) for v in result.values())
    # the same draws again, eagerly, batch by batch: candidates, scores, hit flags
    s.rng.state.copy_(st)
    trainer.use_graph = False
    kmax = max(trainer.topk)
    recs_e, recs_o = [], []
    model.eval()
    with torch.no_grad():
        for inter, _, _, pos in loader:
            inter = inter.to('cuda')
            pos = pos.cuda()
            cand = torch.empty((len(pos), 101), dtype=torch.int64, device='cuda')
            s.draw(inter['user_id'], 100, positives=pos, out=cand[:, 1:], ld=101)
            scores, rec = model.sampled_topk(inter, cand, kmax, pos)
            recs_e.append(rec.cpu())
            flags, _, full = NO.sampled_topk(scores.cpu(), cand.cpu(), ds.item_num, kmax)
            lo, hi = NO.sampled_rank_bounds(full, pos.cpu(), tol=2e-6 * float(scores.abs().max()))
            r = NO.flags_rank(rec.cpu(), kmax)
            assert bool(((r >= lo.clamp(max=kmax)) & (r <= hi.clamp(max=kmax))).all())
            recs_o.append(torch.cat((flags, torch.ones_like(flags[:, :1])), 1))
    rec_e = torch.cat(recs_e)
    # graphed and eager evaluation give identical rec for identical sampler state
    s.rng.state.copy_(st)
    trainer.use_graph = True
    rec_g = torch.cat([trainer.eval_batch(b, neg_sampler=s, neg_num=100).cpu() for b in loader])
    assert torch.equal(rec_g, rec_e)
    want = trainer.evaluator.evaluate(torch.cat(recs_o).numpy())
    for k, v in want.items():
        assert abs(result[k] - v) <= 1e-4, (k, result[k], v)


def test_one_trainer_replays_each_samplers_own_graph(A):
    """two loaders with different samplers (uniform and popularity, different phases) evaluated alternately on ONE trainer: each
    graphed pass draws from its own sampler -- the same rec as the eager path from the same sampler state -- and a packed loader
    batch reaches the captured graph as one copy"""
    config, ds, loader_u, model, trainer = _synthetic_c2(A, 'ACSASRec', 'uniform')
    f = ds.inter_feat
    off, items = A.ops.used_item_csr(f['user_id'].numpy(), f['item_id'].numpy(), len(ds) + 1, ds.item_num)
    sp = A.ops.NegSampler('popularity', off, items, ds.item_num, seed=42, phase=2,
                          counts=np.bincount(f['item_id'].numpy(), minlength=ds.item_num))
    loader_p = A.data.NegSampleEvalDataLoader(config, ds, sp, 100)
    model.eval()
    recs = {}
    for loader in (loader_u, loader_p, loader_u, loader_p):
        s = loader.neg_sampler
        s.to_device('cuda')
        st = s.rng.state.clone()
        trainer.use_graph = True
        rec_g = torch.cat([trainer.eval_batch(b, neg_sampler=s, neg_num=100).cpu() for b in loader])
        s.rng.state.copy_(st)
        trainer.use_graph = False
        rec_e = torch.cat([trainer.eval_batch(b, neg_sampler=s, neg_num=100).cpu() for b in loader])
        assert torch.equal(rec_g, rec_e), s.distribution
        recs.setdefault(s.distribution, []).append(rec_g)
    assert not torch.equal(recs['uniform'][0], recs['popularity'][0])
    graphs = [g for k, g in trainer._eval_graphs.items() if k[0] == 'sampled']
    assert len(graphs) == 2 and {id(g['sampler']) for g in graphs} == {id(loader_u.neg_sampler), id(sp)}
    batch = next(iter(loader_u))
    loader_u.pr = 0
    assert any(g['inter'].layout == batch[0].layout for g in graphs)          # one-copy input path


def test_popularity_fallback_for_the_heaviest_user_is_the_documented_mixture(A, ml100k):
    """the bounded alias retries (16) give way to the uniform-complement draw with probability f^16, f = the popularity mass of
    the user's used set.  For the heaviest ml-100k user f = 0.70 (0.33 % of its draws); the draws follow exactly
    (1 - f^16) * popularity-restricted + f^16 * uniform-complement"""
    from scipy.stats import chisquare
    config, ds, splits = ml100k
    s = A.dataset.build_neg_samplers(config, splits, None, 'popularity')[2]
    p_all = s.counts / s.counts.sum()
    mass = np.array([p_all[s.used_items[s.used_offsets[u]:s.used_offsets[u + 1]]].sum() for u in range(s.n_users)])
    u = int(np.argmax(mass))
    fb = mass[u] ** 16
    assert 0.6 < mass[u] < 0.75 and fb < 5e-3
    used = set(s.used_items[s.used_offsets[u]:s.used_offsets[u + 1]].tolist())
    comp = np.array([i for i in range(1, ds.item_num) if i not in used])
    many = draw_many(s, torch.full((1024,), u, dtype=torch.int64, device='cuda'), 256, reps=4).reshape(-1).numpy()
    assert not np.isin(many, list(used)).any()
    p = (1 - fb) * s.counts[comp] / s.counts[comp].sum() + fb / len(comp)
    cnt = np.bincount(many, minlength=ds.item_num)[comp].astype(np.float64)
    keep = p * many.size >= 5
    exp = p[keep] * many.size
    exp *= cnt[keep].sum() / exp.sum()
    assert chisquare(cnt[keep], exp).pvalue > 1e-4
    # never-a-target items are reached only through the fallback: their share matches f^16 * (their part of the complement)
    zero = s.counts[comp] == 0
    want = many.size * fb * zero.sum() / len(comp)
    assert abs(cnt[zero].sum() - want) < 6 * np.sqrt(want) + 5


def test_sampled_evaluation_leaves_training_rng_untouched(A, tmp_path):
    states = []
    for mode in ('full', 'uni100'):
        config = ml100k_config(A, checkpoint_dir=str(tmp_path),
                               eval_args={'split': {'LS': 'valid_and_test'}, 'group_by': 'user', 'order': 'TO', 'mode': mode})
        ds = A.create_dataset(config)
        tr, va, te = A.data_preparation(config, ds)
        torch.manual_seed(0)
        model = A.ACSASRec(config, tr.dataset).cuda()
        trainer = A.ACSASRecTrainer(config, model)
        trainer._train_epoch(tr, 0)
        res = trainer.evaluate(va, load_best_model=False)
        trainer._train_epoch(tr, 1)
        assert all(np.isfinite(v) for v in res.values())
        states.append(model._rng.state.cpu().clone())
    assert torch.equal(states[0], states[1])


# ---- BPR with sampled negatives ---------------------------------------------------------------------------------
def _bpr_setup(A, name, device_resident, tmp_path):
    cfg = O.default_cfg(loss_type='BPR', hidden_dropout_prob=0.0, attn_dropout_prob=0.0)
    cfg.update(time_span=64, user_hidden_size=32, item_hidden_size=32)
    B, V = 64, 400
    config = make_config(A, cfg, model=name, train_batch_size=B, checkpoint_dir=str(tmp_path), device_resident_data=device_resident)
    ds = A.data.SyntheticSequentialDataset(config, 2 * B, V, seed=21)
    f = ds.inter_feat
    off, items = A.ops.used_item_csr(f['user_id'].numpy(), f['item_id'].numpy(), 2 * B + 1, V)
    s = A.ops.NegSampler('uniform', off, items, V, seed=42)
    torch.manual_seed(4)
    model = getattr(A, name)(config, ds).cuda()
    params = {k: v.detach().clone() for k, v in model.state_dict().items()}
    return config, ds, s, model, params


@pytest.mark.parametrize('name,device_resident', [('ACSASRec', True), ('ACSASRec', False), ('ACSSEPT', False)])
def test_bpr_step_with_sampled_negatives_equals_explicit_negatives(A, tmp_path, name, device_resident):
    """one captured BPR step whose negatives the sampler draws (inside the DeviceTrainDataLoader's gather, or into the static
    neg slot of a host batch) equals the existing BPR step fed the same negatives as neg_item_id"""
    config, ds, s, model, params = _bpr_setup(A, name, device_resident, tmp_path)
    trainer = getattr(A, name + 'Trainer')(config, model)
    model.train()
    s.to_device('cuda')
    st = s.rng.state.clone()
    if device_resident:
        loader = A.data.DeviceTrainDataLoader(config, ds, shuffle=False, neg_sampler=s)
        loader.new_epoch()
        la, lc = trainer.device_loader_step(loader)
        batch = {k: v[:config['train_batch_size']] for k, v in ds.inter_feat.interaction.items()}
        users, pos = batch['user_id'].cuda(), batch['item_id'].cuda()
    else:
        loader = A.data.TrainDataLoader(config, ds, shuffle=False, neg_sampler=s)
        trainer.train_neg_sampler = s
        host = next(iter(loader))
        la, lc = trainer.graphed_step(host)
        users, pos = host['user_id'].cuda(), host['item_id'].cuda()
    torch.cuda.synchronize()
    got = trainer.optimizer.flat_grad.detach().clone()
    # the same negatives, drawn again from the same sampler state, as an explicit field of an eager step on a fresh trainer
    s.rng.state.copy_(st)
    negs = s.draw(users, 1, positives=pos).view(-1)
    model2 = getattr(A, name)(config, ds).cuda()
    model2.load_state_dict(params)
    t2 = getattr(A, name + 'Trainer')(config, model2)
    model2.train()
    f = {k: v[:config['train_batch_size']].cuda() for k, v in ds.inter_feat.interaction.items()}
    f['neg_item_id'] = negs
    la2, lc2 = t2.train_step(A.Interaction(f))
    assert abs(float(la) - float(la2)) <= 1e-5 * abs(float(la2)) + 1e-6
    assert abs(float(lc) - float(lc2)) <= 1e-5 * abs(float(lc2)) + 1e-6
    # gradients (not parameters: Adam's first step turns float-atomic rounding of near-zero gradients into +-lr)
    want = t2.optimizer.flat_grad
    assert float((got - want).abs().max()) <= 1e-4 * float(want.abs().max())


# ---- end to end -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('cfg', ['config/ml-100k-uni100.yaml', 'config/ml-100k-bpr.yaml'])
def test_run_recbole_end_to_end(A, tmp_path, cfg):
    r = subprocess.run([sys.executable, 'run_recbole.py', '--model=ACSASRec', '--dataset=ml-100k', '--config_files=' + cfg,
                        '--epochs=1', '--checkpoint_dir=' + str(tmp_path)], cwd=ROOT, capture_output=True, text=True, timeout=900)
    log = r.stdout + r.stderr
    assert r.returncode == 0, log[-4000:]
    assert 'test result' in log and 'nan' not in log.split('test result')[-1].lower(), log[-2000:]
