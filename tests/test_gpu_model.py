"""End-to-end parity of the CUDA ACSASRec (through the drop-in model / trainer API) against
(a) the golden vectors produced by the real reference and (b) the oracle, plus size-independent
properties at BASELINE.json's full sizes."""
import glob
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import acsr_oracle as O
from golden_util import GOLDEN_DIR, load_case

EVERY = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN_DIR, '*.npz')))
ALL = [n for n in EVERY if not n.startswith(('bert_', 'ssept_', 'ti_', 'oracleonly_'))]      # oracleonly_*: tests/test_oracle_golden.py only
TI = [n for n in EVERY if n.startswith('ti_')]              # ACTiSASRec cases (actisasrec.py on transformer_layers.py)
SSEPT = [n for n in EVERY if n.startswith('ssept_')]        # ACSSEPT cases (acssept.py on transformer_layers.py)
BERT = [n for n in EVERY if n.startswith('bert_')]          # AcBERT4Rec cases (acbert4rec.py)
TRAIN = [n for n in ALL if '_train' in n]
EVAL = [n for n in ALL if '_eval' in n]


@pytest.fixture(scope='module')
def A():
    import ac_tsr_b200 as pkg
    pkg.LIB.load()
    return pkg


class DS:
    def __init__(self, n):
        self.n = n
        self.item_num = n

    def num(self, field):
        return self.n


def make_config(A, cfg, **extra):
    d = dict(cfg)
    d.update(USER_ID_FIELD='user_id', ITEM_ID_FIELD='item_id', LIST_SUFFIX='_list', ITEM_LIST_LENGTH_FIELD='item_length',
             NEG_PREFIX='neg_', device=torch.device('cuda'), seed=42, learning_rate=1e-3, epochs=1, eval_batch_size=256,
             train_batch_size=256, topk=[1, 5, 10, 50], metrics=['Hit', 'MRR', 'NDCG', 'Recall'], valid_metric='Hit@10',
             checkpoint_dir='/tmp/acsr_ckpt', cuda_graph=False)
    d.update(extra)
    return A.Config(model='ACSASRec', config_dict=d)


def build_model(A, c, **extra):
    config = make_config(A, c['cfg'], **extra)
    model = A.ACSASRec(config, DS(c['V'])).to('cuda')
    sd = {k: v.cuda() for k, v in c['params'].items()}
    missing, unexpected = model.load_state_dict(sd, strict=True), None     # reference state_dict loads unchanged
    model._debug_rand = {k: v.cuda() for k, v in c['rand'].d.items()}
    return config, model


def inter_of(A, c):
    b = c['batch']
    f = {'item_id_list': b['item_seq'].cuda(), 'item_length': b['item_len'].cuda(), 'item_id': b['pos'].cuda()}
    if 'neg' in b:                                 # loss_type BPR
        f['neg_item_id'] = b['neg'].cuda()
    return A.Interaction(f)


def rel(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp(min=1e-30))


@pytest.mark.parametrize('name', EVAL)
def test_golden_eval(A, name):
    c = load_case(name)
    z = c['z']
    config, model = build_model(A, c)
    model.eval()
    inter = inter_of(A, c)
    with torch.no_grad():
        att, cal, masks = model.forward(inter['item_id_list'], inter['item_length'])
        assert rel(att, z['out_att']) < 1e-4 and rel(cal, z['out_cal']) < 1e-4
        for l, m in enumerate(masks):
            assert rel(m.pen_sq, z['pen_sq.%d' % l].reshape(1)) < 1e-5
        none, scores = model.full_sort_predict(inter)
        assert none is None and scores.shape == (c['batch']['pos'].shape[0], c['V']) and scores.is_contiguous()
        assert rel(scores, z['scores']) < 1e-4                      # north_star: logits within 1e-3 relative
        val, idx, rec = model.full_sort_topk(inter, c['k'], inter['item_id'])
        ok, nbad = O.topk_equal_modulo_ties(idx.cpu(), torch.from_numpy(z['topk_idx']), torch.from_numpy(z['scores']))
        assert ok, nbad
        assert np.array_equal(rec.cpu().numpy(), z['rec_topk']) or ok
        pa, pc = model.predict(inter)
        assert rel(pa, z['predict_att']) < 1e-4 and rel(pc, z['predict_cal']) < 1e-4
        # the trainer's API-compatible path: scores[:,0] = -inf ; torch.topk
        s2 = scores.view(-1, c['V']).clone()
        s2[:, 0] = -np.inf
        _, idx2 = torch.topk(s2, c['k'], dim=-1)
        ok2, _ = O.topk_equal_modulo_ties(idx2.cpu(), torch.from_numpy(z['topk_idx']), torch.from_numpy(z['scores']))
        assert ok2


@pytest.mark.parametrize('name', TRAIN)
def test_golden_train_losses_and_routed_grads(A, name):
    """reference trainer semantics (trainer.py:672-686) through the drop-in API: .grad after the two backward passes."""
    c = load_case(name)
    z = c['z']
    config, model = build_model(A, c)
    model.train()
    inter = inter_of(A, c)
    l_att, l_cal = model.calculate_loss(inter)
    assert abs(float(l_att) - float(z['loss_att'])) < 1e-4 * abs(float(z['loss_att']))      # north_star: 1e-3
    assert abs(float(l_cal) - float(z['loss_cal'])) < 1e-4 * abs(float(z['loss_cal']))
    for n, p in model.named_parameters():
        p.requires_grad = not ('attack_key_transform' in n or 'attack_query_transform' in n)
    l_cal.backward(retain_graph=True)
    for n, p in model.named_parameters():
        p.requires_grad = ('attack_key_transform' in n or 'attack_query_transform' in n)
    l_att.backward()
    names = [n for n, _ in model.named_parameters()]
    assert set(names) == set(c['grads'])
    for n, p in model.named_parameters():
        ref = c['grads'][n]
        got = p.grad.cpu() if p.grad is not None else torch.zeros_like(ref)
        scale = float(ref.abs().max())
        err = float((got - ref).abs().max())
        assert err <= 1e-3 * scale + 1e-8, (n, err, scale)


@pytest.mark.parametrize('name', ['c1_train', 'beauty_train', 'bpr_train'])
def test_trainer_step_matches_oracle_adam(A, name):
    """one full optimisation step (both losses, routed grads, fused Adam) == oracle grads + oracle Adam."""
    c = load_case(name)
    config, model = build_model(A, c)
    trainer = A.ACSASRecTrainer(config, model)
    model.train()
    la, lc = trainer.train_step(inter_of(A, c))
    b = c['batch']
    _, _, grads = O.train_grads(c['params'], c['cfg'], b['item_seq'], b['item_len'], b['pos'], c['rand'], neg_items=b.get('neg'))
    sd = model.state_dict()
    for n, p0 in c['params'].items():
        want, _, _ = O.adam_step(p0, grads[n], torch.zeros_like(p0), torch.zeros_like(p0), 1, 1e-3)
        got = sd[n].cpu()
        # Adam's first step moves every weight by ~lr*sign(g): compare the update, not the weight
        upd_w, upd_g = (want - p0), (got - p0)
        big = grads[n].abs() > 1e-3 * grads[n].abs().max()
        assert float((upd_w - upd_g)[big].abs().max()) < 2e-5, n
    assert abs(float(lc) - float(c['z']['loss_cal'])) < 1e-4 * abs(float(c['z']['loss_cal']))


def test_graphed_step_equals_eager_step(A):
    """CUDA-graph replay of the step == eager launches (dropout off so both are deterministic)."""
    cfg = O.default_cfg(hidden_dropout_prob=0.0, attn_dropout_prob=0.0)
    V, B, L = 500, 64, 50
    params = O.init_params(cfg, V, seed=1)
    seq, ln, pos = O.synth_batch(B, L, V, seed=5)
    results = []
    for graph in (False, True):
        config = make_config(A, cfg, cuda_graph=graph)
        model = A.ACSASRec(config, DS(V)).to('cuda')
        model.load_state_dict({k: v.cuda() for k, v in params.items()})
        model._debug_rand = {(l, 'noise'): torch.zeros(B, cfg['n_heads'], L, L).cuda() for l in range(cfg['n_layers'])}
        trainer = A.ACSASRecTrainer(config, model)
        model.train()
        inter = A.Interaction({'item_id_list': seq, 'item_length': ln, 'item_id': pos})
        losses = []
        for _ in range(3):
            la, lc = trainer.graphed_step(inter) if graph else trainer.train_step(inter.to('cuda'))
            losses.append((float(la), float(lc)))
        results.append((losses, {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}))
    (l0, s0), (l1, s1) = results
    for a, b in zip(l0, l1):
        assert abs(a[0] - b[0]) < 1e-4 * abs(a[0]) and abs(a[1] - b[1]) < 1e-4 * abs(a[1])
    assert l0[2][1] < l0[0][1]                      # the calibrated loss goes down
    for k in s0:
        assert float((s0[k] - s1[k]).abs().max()) < 1e-5, k


def test_full_size_properties_beauty_shape(A):
    """BASELINE config #2 (V=12,102, L=50, d=64, N=2, B=256): properties that need no CPU reference."""
    cfg = O.default_cfg()
    V, B, L, k = 12102, 256, 50, 50
    config = make_config(A, cfg)
    torch.manual_seed(42)
    model = A.ACSASRec(config, DS(V)).to('cuda')
    seq, ln, pos = O.synth_batch(B, L, V, seed=42)
    inter = A.Interaction({'item_id_list': seq.cuda(), 'item_length': ln.cuda(), 'item_id': pos.cuda()})
    model.eval()
    with torch.no_grad():
        _, scores = model.full_sort_predict(inter)
        val, idx, rec = model.full_sort_topk(inter, k, inter['item_id'])
    s = scores.clone()
    s[:, 0] = -np.inf
    rv, ri = torch.topk(s, k, dim=-1)
    assert (val[:, :-1] >= val[:, 1:]).all()                              # sortedness
    ok, nbad = O.topk_equal_modulo_ties(idx.cpu(), ri.cpu(), scores.cpu())
    assert ok, nbad                                                       # fused top-k == materialised top-k
    assert torch.equal(rec[:, :-1].bool().cpu(), (idx == inter['item_id'].view(-1, 1)).cpu())
    # CE identity: loss == logsumexp(scores) - scores[target], softmax-gradient rows sum to zero
    out, _ = model._encode(inter['item_id_list'], inter['item_length'], need_attacked=False)
    out = out.detach().requires_grad_(True)
    E = model.item_embedding.weight
    loss = A.ops.LogitsCEFn.apply(out, E, inter['item_id'], 1, 3)[0]
    ref = (torch.logsumexp(scores.double(), 1) - scores.double()[torch.arange(B), inter['item_id']]).mean()
    assert abs(float(loss) - float(ref)) < 1e-5 * abs(float(ref))
    lse = torch.logsumexp(scores.double(), 1).float()
    Gt = A.ops.ce_grad_matrix_t(out.detach(), E.detach(), lse, inter['item_id'], torch.ones(B).cuda(), 3)
    assert float(Gt.double().sum(0).abs().max()) < 1e-4
    # a padded-key change must not leak: padding positions never influence the calibrated output
    seq2 = seq.clone()
    rows = torch.arange(B)
    with torch.no_grad():
        out_a, _ = model._encode(seq.cuda(), ln.cuda(), need_attacked=False)
        short = ln < L
        seq3 = seq.clone()
        seq3[short, -1] = 0                                               # already 0: idempotent
        out_b, _ = model._encode(seq3.cuda(), ln.cuda(), need_attacked=False)
    assert torch.equal(out_a, out_b)


def test_checkpoint_roundtrip_and_eval_loop(A, tmp_path):
    cfg = O.default_cfg(n_layers=1)
    V, L = 400, 50
    config = make_config(A, cfg, checkpoint_dir=str(tmp_path), epochs=1, train_batch_size=64, eval_batch_size=64,
                         cuda_graph=True)
    torch.manual_seed(0)
    train_ds = A.data.SyntheticSequentialDataset(config, 64 * 3 + 10, V, seed=1)
    valid_ds = A.data.SyntheticSequentialDataset(config, 100, V, seed=2)
    model = A.ACSASRec(config, train_ds).to('cuda')
    trainer = A.ACSASRecTrainer(config, model)
    trainer.epochs = 1
    train_loader = A.data.TrainDataLoader(config, train_ds, shuffle=True)
    valid_loader = A.data.FullSortEvalDataLoader(config, valid_ds)
    # fit() runs range(0, 2*epochs) epochs (trainer.py:835); the last batch (10 rows) takes the eager path
    score, result = trainer.fit(train_loader, valid_loader, verbose=False, saved=True)
    assert set(result) == {'%s@%d' % (m, k) for m in ('hit', 'mrr', 'ndcg', 'recall') for k in (1, 5, 10, 50)}
    assert os.path.exists(trainer.saved_model_file)
    ck = torch.load(trainer.saved_model_file, map_location='cpu', weights_only=False)
    assert set(ck) == {'config', 'epoch', 'cur_step', 'best_valid_score', 'state_dict', 'other_parameter', 'optimizer'}
    res2 = trainer.evaluate(valid_loader, load_best_model=True)
    trainer.fused_topk = False                     # API-compatible path: full_sort_predict + scores[:,0]=-inf + topk
    res3 = trainer.evaluate(valid_loader, load_best_model=False)
    for k in res2:
        assert abs(res2[k] - res3[k]) <= 1e-4      # north_star: Recall@10 / NDCG@10 within 1e-4
    # metrics equal the oracle's restatement of metrics.py
    trainer.fused_topk = True
    model.eval()
    recs = torch.cat([trainer.eval_batch(b) for b in valid_loader]).cpu().numpy()
    want = O.topk_metrics(recs[:, :-1], recs[:, -1], topk=(1, 5, 10, 50))
    for k, v in res2.items():
        assert abs(want[k] - v) < 1e-9


@pytest.mark.parametrize('name', TRAIN)
def test_fused_step_matches_reference_grads(A, name):
    """the explicit two-stream step (fused_step.py) against the reference's losses and routed .grad."""
    c = load_case(name)
    z = c['z']
    config, model = build_model(A, c)
    trainer = A.ACSASRecTrainer(config, model)            # FlatAdam: parameters / grads become views of flat buffers
    assert trainer.fused is not None
    model.train()
    l_att, l_cal = trainer.fused(inter_of(A, c))
    assert abs(float(l_att) - float(z['loss_att'])) < 1e-4 * abs(float(z['loss_att']))
    assert abs(float(l_cal) - float(z['loss_cal'])) < 1e-4 * abs(float(z['loss_cal']))
    for n, p in model.named_parameters():
        ref = c['grads'][n]
        got = p.grad.cpu()
        scale = float(ref.abs().max())
        err = float((got - ref).abs().max())
        assert err <= 1e-3 * scale + 1e-8, (n, err, scale)


def test_fused_step_equals_autograd_step_full_batch(A):
    """B=256 Beauty shape, dropout on (Philox): fused explicit step vs autograd path cannot share masks
    (different stream layout), so compare with dropout off and injected zero noise."""
    cfg = O.default_cfg(hidden_dropout_prob=0.0, attn_dropout_prob=0.0)
    V, B, L = 12102, 256, 50
    params = O.init_params(cfg, V, seed=3)
    seq, ln, pos = O.synth_batch(B, L, V, seed=6)
    grads = []
    for fused in (False, True):
        config = make_config(A, cfg, fused_step=fused)
        model = A.ACSASRec(config, DS(V)).to('cuda')
        model.load_state_dict({k: v.cuda() for k, v in params.items()})
        g = torch.Generator().manual_seed(0)
        model._debug_rand = {(l, 'noise'): torch.randn(B, cfg['n_heads'], L, L, generator=g).cuda() for l in range(cfg['n_layers'])}
        trainer = A.ACSASRecTrainer(config, model)
        assert (trainer.fused is not None) == fused
        model.train()
        inter = A.Interaction({'item_id_list': seq.cuda(), 'item_length': ln.cuda(), 'item_id': pos.cuda()})
        if fused:
            la, lc = trainer.fused(inter)
        else:
            trainer.optimizer.zero_grad()
            la, lc = model.calculate_loss(inter)
            trainer._route(attack=False); lc.backward(retain_graph=True)
            trainer._route(attack=True); la.backward()
        grads.append((float(la), float(lc), {n: p.grad.detach().cpu().clone() for n, p in model.named_parameters()}))
    (a0, c0, g0), (a1, c1, g1) = grads
    assert abs(a0 - a1) < 1e-5 * abs(a0) and abs(c0 - c1) < 1e-5 * abs(c0)
    for n in g0:
        scale = float(g0[n].abs().max())
        assert float((g0[n] - g1[n]).abs().max()) <= 2e-4 * scale + 1e-9, n


@pytest.mark.parametrize('nb', [2, 4])
def test_fused_step_branches_equal_single_chain(A, nb):
    """the step cut into nb parallel sequence groups == the single chain (dropout off, injected noise)."""
    cfg = O.default_cfg(hidden_dropout_prob=0.0, attn_dropout_prob=0.0)
    V, B, L = 3001, 64, 50
    params = O.init_params(cfg, V, seed=3)
    seq, ln, pos = O.synth_batch(B, L, V, seed=6)
    res = []
    for branches in (1, nb):
        config = make_config(A, cfg, fused_step=True)
        model = A.ACSASRec(config, DS(V)).to('cuda')
        model.load_state_dict({k: v.cuda() for k, v in params.items()})
        g = torch.Generator().manual_seed(0)
        model._debug_rand = {(l, 'noise'): torch.randn(B, cfg['n_heads'], L, L, generator=g).cuda() for l in range(cfg['n_layers'])}
        trainer = A.ACSASRecTrainer(config, model)
        trainer.fused.n_branches = branches
        model.train()
        inter = A.Interaction({'item_id_list': seq.cuda(), 'item_length': ln.cuda(), 'item_id': pos.cuda()})
        la, lc = trainer.fused(inter)
        torch.cuda.synchronize()
        res.append((float(la), float(lc), trainer.optimizer.flat_grad.detach().cpu().clone()))
    (a0, c0, g0), (a1, c1, g1) = res
    assert abs(a0 - a1) < 1e-5 * abs(a0) and abs(c0 - c1) < 1e-5 * abs(c0)
    assert float((g0 - g1).abs().max()) <= 1e-4 * float(g0.abs().max())


def test_full_size_properties_million_item_catalogue(A):
    """BASELINE config #4 shape on one GPU (V=1,000,001, B=256): fused CE and fused top-k against the
    materialised scores of the same device GEMM (size-independent identities, no CPU reference needed)."""
    V, B, k = 1000001, 256, 50
    g = torch.Generator().manual_seed(4)
    out = (torch.randn(2 * B, 64, generator=g) * 0.7).cuda()
    E = (torch.randn(V, 64, generator=g) * 0.05).cuda()
    tgt = torch.randint(1, V, (2 * B,), generator=g).cuda()
    scores = A.ops.logits_scores(out, E, 3)                                 # [512, 1e6] fp32 = 2 GB
    chk = (out[:8].double() @ E[:4096].double().t())
    assert float((scores[:8, :4096].double() - chk).abs().max()) < 2e-6 * float(chk.abs().max())
    loss = A.ops.LogitsCEFn.apply(out, E, tgt, 2, 3)
    ref = torch.logsumexp(scores.double(), 1) - scores.double()[torch.arange(2 * B), tgt]
    want = torch.stack([ref[:B].mean(), ref[B:].mean()])
    assert float((loss.double() - want).abs().max()) < 1e-5 * float(want.abs().max())
    val, idx, rec = A.ops.full_sort_topk(out[:B], E, k, tgt[:B], 3)
    s = scores[:B].clone()
    s[:, 0] = -np.inf
    rv, ri = torch.topk(s, k, dim=-1)
    ok, nbad = O.topk_equal_modulo_ties(idx.cpu(), ri.cpu(), scores[:B].cpu())
    assert ok, nbad
    assert (val[:, :-1] >= val[:, 1:]).all()
    assert torch.equal(rec[:, :-1].bool(), idx == tgt[:B].view(-1, 1))
    del scores, s
    # gradient identity: rows of (softmax - onehot) sum to zero, d_out = G.E
    lse = torch.logsumexp(A.ops.logits_scores(out[:64], E, 3).double(), 1).float()
    Gt = A.ops.ce_grad_matrix_t(out[:64].contiguous(), E, lse, tgt[:64].contiguous(), torch.ones(64).cuda(), 3)
    assert float(Gt.double().sum(0).abs().max()) < 1e-4
    d_out, _ = A.ops.linear_wgrad(Gt, E, want_bias=False)
    want_d = (Gt.double().t() @ E.double())
    assert float((d_out.double() - want_d).abs().max()) < 1e-4 * float(want_d.abs().max())


SHAPES = {
    # BASELINE.json configs at their own model shapes, small batch / catalogue so the CPU oracle finishes in seconds
    'c3_yelp_variant': (dict(n_layers=3, n_heads=8, hidden_size=128, inner_size=64), 2003, 6),          # config/yelp.yaml:39-42
    'c5_long_stress': (dict(n_layers=4, n_heads=4, hidden_size=256, inner_size=1024, MAX_ITEM_LIST_LENGTH=200), 1201, 3),
    'c5_long_fixed': (dict(n_layers=2, n_heads=4, hidden_size=256, inner_size=512, MAX_ITEM_LIST_LENGTH=200,
                           combine_option='fixed', two_level=False, rich_calibrated_combine='fixed'), 301, 2),
    # hidden size 64 at inner sizes that are not multiples of 64: the tensor-core step without acsr_dense_bwd (six launches for
    # the first layer's dense backward), with the fused last-layer tail (96) and without it (100, not a multiple of 16)
    'inner96': (dict(n_layers=2, inner_size=96), 2003, 6),
    'inner100': (dict(n_layers=2, inner_size=100), 2003, 6),
}


@pytest.mark.parametrize('shape', sorted(SHAPES))
def test_config_shapes_train_step_and_eval_vs_oracle(A, shape):
    """fused training step (losses + routed gradients) and full-sort eval against the oracle on seeded inputs with the
    dropout masks / attack noise injected, at the model shapes of BASELINE configs #3 (repo variant) and #5 and at hidden
    size 64 with inner sizes that take the step's other tensor-core paths."""
    kw, V, B = SHAPES[shape]
    cfg = O.default_cfg(**kw)
    L, N, H = cfg['MAX_ITEM_LIST_LENGTH'], cfg['n_layers'], cfg['n_heads']
    params = O.init_params(cfg, V, seed=7)
    g = torch.Generator().manual_seed(8)
    for n in params:                               # non-trivial biases / LayerNorm weights
        if n.endswith('.bias'):
            params[n] = params[n] + torch.randn(params[n].shape, generator=g) * 0.02
    seq, ln, pos = O.synth_batch(B, L, V, seed=9)
    ln[0] = L
    seq[0] = torch.randint(1, V, (L,), generator=g)
    rnd = O.draw_rand(cfg, B, L, seed=10, train=True)
    la_o, lc_o, grads = O.train_grads(params, cfg, seq, ln, pos, rnd)
    config = make_config(A, cfg)
    model = A.ACSASRec(config, DS(V)).to('cuda')
    model.load_state_dict({k: v.cuda() for k, v in params.items()}, strict=True)
    model._debug_rand = {k: v.cuda() for k, v in rnd.d.items()}
    trainer = A.ACSASRecTrainer(config, model)
    assert trainer.fused is not None
    model.train()
    inter = A.Interaction({'item_id_list': seq.cuda(), 'item_length': ln.cuda(), 'item_id': pos.cuda()})
    la, lc = trainer.fused(inter)
    assert abs(float(la) - float(la_o)) < 1e-4 * abs(float(la_o)), (float(la), float(la_o))      # north_star: 1e-3
    assert abs(float(lc) - float(lc_o)) < 1e-4 * abs(float(lc_o)), (float(lc), float(lc_o))
    for n, p in model.named_parameters():
        ref = grads[n]
        scale = float(ref.abs().max())
        err = float((p.grad.cpu() - ref).abs().max())
        assert err <= 1e-3 * scale + 1e-8, (n, err, scale)
    # eval: scores, top-k indices (modulo ties), hit flags
    model.eval()
    model._debug_rand = None
    k = 50
    with torch.no_grad():
        _, scores = model.full_sort_predict(inter)
        val, idx, rec = model.full_sort_topk(inter, k, inter['item_id'])
    ref_scores = O.full_sort_scores(params, cfg, seq, ln)
    assert rel(scores, ref_scores) < 1e-4
    _, ref_idx = O.full_sort_topk(ref_scores, k)
    ok, nbad = O.topk_equal_modulo_ties(idx.cpu(), ref_idx, ref_scores)
    assert ok, nbad
    assert torch.equal(rec.cpu()[:, :-1], O.hit_flags(idx.cpu(), pos))


def test_resume_from_reference_format_checkpoint(A, tmp_path):
    """trainer.py:733-761: a checkpoint whose 'optimizer' entry is torch.optim.Adam's state_dict (what the reference writes)
    resumes in this trainer: the step after the resume equals the step of an uninterrupted run (dropout off)."""
    cfg = O.default_cfg(hidden_dropout_prob=0.0, attn_dropout_prob=0.0, n_layers=1)
    V, B, L = 300, 32, 50
    params = O.init_params(cfg, V, seed=2)
    seq, ln, pos = O.synth_batch(B, L, V, seed=3)

    def fresh():
        config = make_config(A, cfg, checkpoint_dir=str(tmp_path))
        model = A.ACSASRec(config, DS(V)).to('cuda')
        model.load_state_dict({k: v.cuda() for k, v in params.items()})
        model._debug_rand = {(l, 'noise'): torch.zeros(B, cfg['n_heads'], L, L).cuda() for l in range(cfg['n_layers'])}
        trainer = A.ACSASRecTrainer(config, model)
        model.train()
        return model, trainer
    inter = A.Interaction({'item_id_list': seq.cuda(), 'item_length': ln.cuda(), 'item_id': pos.cuda()})
    m1, t1 = fresh()
    t1.train_step(inter)
    t1._save_checkpoint(0, verbose=False)
    ck = torch.load(t1.saved_model_file, map_location='cpu', weights_only=False)
    assert set(ck['optimizer']) == {'state', 'param_groups'}                     # torch.optim.Adam's layout
    ref_adam = torch.optim.Adam([torch.nn.Parameter(p.detach().cpu().clone()) for p in m1.parameters()], lr=1e-3)
    ref_adam.load_state_dict(ck['optimizer'])                                    # the reference trainer's resume_checkpoint does this
    t1.train_step(inter)
    m2, t2 = fresh()
    t2.resume_checkpoint(t1.saved_model_file)
    assert t2.start_epoch == 1
    m2.train()
    t2.train_step(inter)
    for (n, a), (_, b) in zip(m1.state_dict().items(), m2.state_dict().items()):
        assert float((a - b).abs().max()) < 1e-6, n


def test_annealing_schedule_advances_through_the_graph_path(A):
    """combine_option 'annealing' (layers.py:889-891): the rate is a host float that changes every forward; graphed_step must not
    freeze it (such models launch eagerly) and the warm-up of a capture must not advance it."""
    cfg = O.default_cfg(hidden_dropout_prob=0.0, attn_dropout_prob=0.0, combine_option='annealing', n_layers=2)
    V, B, L = 300, 16, 50
    params = O.init_params(cfg, V, seed=4)
    seq, ln, pos = O.synth_batch(B, L, V, seed=5)
    res = []
    for graph in (False, True):
        config = make_config(A, cfg, cuda_graph=graph)
        model = A.ACSASRec(config, DS(V)).to('cuda')
        model.load_state_dict({k: v.cuda() for k, v in params.items()})
        for layer in model.trm_encoder.layer:
            layer.anneal_step = 70000                                            # exp(-0.7): far from both ends
        model._debug_rand = {(l, 'noise'): torch.zeros(B, cfg['n_heads'], L, L).cuda() for l in range(cfg['n_layers'])}
        trainer = A.ACSASRecTrainer(config, model)
        model.train()
        inter = A.Interaction({'item_id_list': seq, 'item_length': ln, 'item_id': pos})
        losses = []
        for _ in range(3):
            la, lc = trainer.graphed_step(inter) if graph else trainer.train_step(inter.to('cuda'))
            losses.append((float(la), float(lc)))
        assert [layer.anneal_step for layer in model.trm_encoder.layer] == [70003, 70003]
        model.eval()
        with torch.no_grad():
            trainer.eval_batch((inter.to('cuda'), None, None, pos.cuda()))
        assert [layer.anneal_step for layer in model.trm_encoder.layer] == [70004, 70004]
        res.append(losses)
    for a, b in zip(*res):
        assert abs(a[0] - b[0]) < 1e-5 * abs(a[0]) and abs(a[1] - b[1]) < 1e-5 * abs(a[1])
    # and the rate really enters the result: the oracle with the same three rates reproduces the first loss
    import math
    rates = [math.exp(-70000 / 100000)] * cfg['n_layers']
    rnd = O.Rand({(l, 'noise'): torch.zeros(B, cfg['n_heads'], L, L) for l in range(cfg['n_layers'])})
    la_o, lc_o, _ = O.train_grads(params, cfg, seq, ln, pos, rnd, anneal_rates=rates)
    assert abs(res[0][0][1] - float(lc_o)) < 1e-4 * abs(float(lc_o))


def test_device_resident_loader_epoch_equals_host_loader_steps(A):
    """f-2: the HBM-resident loader (on-device permutation, batch gathered INSIDE the captured step) trains exactly like the
    same batches fed one by one: every row of the epoch exactly once, same parameters after the epoch (dropout off)."""
    cfg = O.default_cfg(hidden_dropout_prob=0.0, attn_dropout_prob=0.0, n_layers=1)
    V, L, B, n = 300, 50, 32, 32 * 5 + 7                      # five full batches + a ragged tail of 7 rows
    params = O.init_params(cfg, V, seed=2)

    def fresh(graph):
        config = make_config(A, cfg, train_batch_size=B, cuda_graph=graph, seed=123)
        ds = A.data.SyntheticSequentialDataset(config, n, V, seed=5)
        model = A.ACSASRec(config, ds).to('cuda')
        model.load_state_dict({k: v.cuda() for k, v in params.items()})
        model._debug_rand = {(l, 'noise'): torch.zeros(B, cfg['n_heads'], L, L).cuda() for l in range(cfg['n_layers'])}
        trainer = A.ACSASRecTrainer(config, model)
        model.train()
        return config, ds, model, trainer
    config, ds, m1, t1 = fresh(True)
    loader = A.data.DeviceTrainDataLoader(config, ds, shuffle=True)
    # iterating the loader yields every row exactly once, in the order of its device permutation
    seen = torch.cat([b['item_id'].cpu() for b in loader])
    perm = loader.perm.cpu()
    assert torch.equal(seen, ds.inter_feat['item_id'][perm]) and sorted(perm.tolist()) == list(range(n))
    assert not torch.equal(perm, torch.arange(n))
    # epoch through the trainer: graph replays that gather their own batch + eager tail
    loader.gen.manual_seed(77)
    la, lc = t1._train_epoch(loader, 0)
    assert t1._dgraph is not None and int(loader.cursor.item()) == n // B
    perm = loader.perm.cpu()
    # the same batches, one eager step each, from host tensors
    config2, ds2, m2, t2 = fresh(False)
    m2._debug_rand = None
    tot_c = 0.0
    feat = ds2.inter_feat
    for i in range(0, n, B):
        idx = perm[i:i + B]
        rows = len(idx)
        m2._debug_rand = {(l, 'noise'): torch.zeros(rows, cfg['n_heads'], L, L).cuda() for l in range(cfg['n_layers'])}
        inter = A.Interaction({k: feat[k][idx].cuda() for k in ('item_id_list', 'item_length', 'item_id')})
        _, c = t2.train_step(inter)
        tot_c += float(c)
    assert abs(lc - tot_c) < 1e-4 * abs(tot_c), (lc, tot_c)
    for (k, a), (_, b) in zip(m1.state_dict().items(), m2.state_dict().items()):
        assert float((a - b).abs().max()) < 2e-5, k
    # a second epoch draws a new permutation and rewinds the cursor
    t1._train_epoch(loader, 1)
    assert not torch.equal(loader.perm.cpu(), perm) and int(loader.cursor.item()) == n // B


# ---- AcBERT4Rec (SURVEY section 8 f-4): goldens from the real reference (tests/golden/make_golden.py: make_bert_case) ----
def build_bert(A, c, **extra):
    cfg = dict(c['cfg'])
    config = make_config(A, cfg, **extra)
    model = A.AcBERT4Rec(config, DS(c['V'])).to('cuda')
    model.load_state_dict({k: v.cuda() for k, v in c['params'].items()}, strict=True)      # reference state_dict loads unchanged
    model._debug_rand = {k: v.cuda() for k, v in c['rand'].d.items()}
    return config, model


@pytest.mark.parametrize('name', [n for n in BERT if '_train' in n])
def test_bert_golden_train_losses_and_routed_grads(A, name):
    c = load_case(name)
    z, b = c['z'], c['batch']
    config, model = build_bert(A, c)
    assert tuple(model.item_embedding.weight.shape) == (c['V'] + 1, c['cfg']['hidden_size'])
    model._debug_masked = tuple(b[k].cuda() for k in ('masked_seq', 'pos_items', 'neg_items', 'masked_index'))
    model.train()
    l_att, l_cal = model.calculate_loss(inter_of(A, c))
    assert abs(float(l_att) - float(z['loss_att'])) < 1e-4 * abs(float(z['loss_att']))
    assert abs(float(l_cal) - float(z['loss_cal'])) < 1e-4 * abs(float(z['loss_cal']))
    for n, p in model.named_parameters():
        p.requires_grad = not ('attack_key_transform' in n or 'attack_query_transform' in n)
    l_cal.backward(retain_graph=True)
    for n, p in model.named_parameters():
        p.requires_grad = ('attack_key_transform' in n or 'attack_query_transform' in n)
    l_att.backward()
    assert set(n for n, _ in model.named_parameters()) == set(c['grads'])
    for n, p in model.named_parameters():
        ref = c['grads'][n]
        got = p.grad.cpu() if p.grad is not None else torch.zeros_like(ref)
        scale = float(ref.abs().max())
        err = float((got - ref).abs().max())
        assert err <= 1e-3 * scale + 1e-8, (n, err, scale)


@pytest.mark.parametrize('name', [n for n in BERT if '_eval' in n])
def test_bert_golden_eval(A, name):
    c = load_case(name)
    z = c['z']
    config, model = build_bert(A, c)
    model.eval()
    inter = inter_of(A, c)
    with torch.no_grad():
        sa, sc = model.full_sort_predict(inter)
        assert rel(sc, z['scores']) < 1e-4 and rel(sa, z['scores_att']) < 1e-4
        assert sc.shape == (c['batch']['pos'].shape[0], c['V'])
        val, idx, rec = model.full_sort_topk(inter, c['k'], inter['item_id'])
        ok, nbad = O.topk_equal_modulo_ties(idx.cpu(), torch.from_numpy(z['topk_idx']), torch.from_numpy(z['scores']))
        assert ok, nbad
        pa, pc = model.predict(inter)
        assert rel(pa, z['predict_att']) < 1e-4 and rel(pc, z['predict_cal']) < 1e-4


def test_bert_gate_cannot_be_evaluated_like_the_reference(A):
    """combine_option gate: Linear(hidden, 50) against the 51 positions of reconstruct_test_data -- a shape error in the reference
    (layers.py:887-888), a ValueError here."""
    c = load_case('bert_gate_train')
    config, model = build_bert(A, c)
    model.eval()
    with pytest.raises(ValueError):
        with torch.no_grad():
            model.full_sort_predict(inter_of(A, c))


def test_bert_trainer_epoch_and_eval(A, tmp_path):
    """AcBERT4RecTrainer: the adversarial two-loss step (routed double backward) + full-sort evaluation run end to end"""
    cfg = O.default_cfg(n_layers=1, combine_option='fixed')
    cfg['mask_ratio'] = 0.2
    V = 200
    config = make_config(A, cfg, checkpoint_dir=str(tmp_path), epochs=1, train_batch_size=32, eval_batch_size=32, MAX_ITEM_LIST_LENGTH=49)
    torch.manual_seed(0)
    train_ds = A.data.SyntheticSequentialDataset(config, 32 * 3, V, seed=1)
    valid_ds = A.data.SyntheticSequentialDataset(config, 64, V, seed=2)
    model = A.AcBERT4Rec(config, train_ds).to('cuda')
    trainer = A.AcBERT4RecTrainer(config, model)
    assert trainer.fused is None                      # the autograd path over the same kernels
    before = model.item_embedding.weight.detach().clone()
    score, result = trainer.fit(A.data.TrainDataLoader(config, train_ds, shuffle=True), A.data.FullSortEvalDataLoader(config, valid_ds),
                                verbose=False, saved=True)
    assert float((model.item_embedding.weight.detach() - before).abs().max()) > 0
    assert all(np.isfinite(v) for v in result.values()) and 'hit@10' in result


# ---- ACSSEPT (SURVEY section 8 f-4): goldens from the real reference (tests/golden/make_golden.py: make_ssept_case) ----
class DSU:
    def __init__(self, n_items, n_users):
        self.n_items, self.n_users, self.item_num = n_items, n_users, n_items

    def num(self, field):
        return self.n_users if field == 'user_id' else self.n_items


def build_ssept(A, c, **extra):
    config = make_config(A, dict(c['cfg']), **extra)
    config['model'] = 'ACSSEPT'
    model = A.ACSSEPT(config, DSU(c['V'], int(c['z']['U']))).to('cuda')
    model.load_state_dict({k: v.cuda() for k, v in c['params'].items()}, strict=True)      # reference state_dict loads unchanged
    model._debug_rand = {k: v.cuda() for k, v in c['rand'].d.items()}
    return config, model


def ssept_inter(A, c):
    inter = inter_of(A, c)
    inter.interaction['user_id'] = c['batch']['user'].cuda()
    return inter


@pytest.mark.parametrize('name', [n for n in SSEPT if '_train' in n])
def test_ssept_golden_train_losses_and_routed_grads(A, name):
    c = load_case(name)
    z = c['z']
    config, model = build_ssept(A, c)
    assert model.hidden_size == c['cfg']['item_hidden_size'] + c['cfg']['user_hidden_size']
    model.train()
    l_att, l_cal = model.calculate_loss(ssept_inter(A, c))
    assert abs(float(l_att) - float(z['loss_att'])) < 1e-4 * abs(float(z['loss_att']))
    assert abs(float(l_cal) - float(z['loss_cal'])) < 1e-4 * abs(float(z['loss_cal']))
    for n, p in model.named_parameters():
        p.requires_grad = not ('attack_key_transform' in n or 'attack_query_transform' in n)
    l_cal.backward(retain_graph=True)
    for n, p in model.named_parameters():
        p.requires_grad = ('attack_key_transform' in n or 'attack_query_transform' in n)
    l_att.backward()
    assert set(n for n, _ in model.named_parameters()) == set(c['grads'])
    for n, p in model.named_parameters():
        ref = c['grads'][n]
        got = p.grad.cpu() if p.grad is not None else torch.zeros_like(ref)
        scale = float(ref.abs().max())
        err = float((got - ref).abs().max())
        # the reference's own gradient of user_embedding through the loss is rounding noise around an exact zero (a per-row
        # constant added to every logit): compare against the scale of the whole tensor
        assert err <= 1e-3 * scale + 1e-7, (n, err, scale)


@pytest.mark.parametrize('name', [n for n in SSEPT if '_eval' in n])
def test_ssept_golden_eval(A, name):
    c = load_case(name)
    z = c['z']
    config, model = build_ssept(A, c)
    model.eval()
    inter = ssept_inter(A, c)
    with torch.no_grad():
        att, cal, masks = model.forward(inter['item_id_list'], inter['item_length'], inter['user_id'])
        assert rel(att, z['out_att']) < 1e-4 and rel(cal, z['out_cal']) < 1e-4
        for l, m in enumerate(masks):
            assert rel(m.pen_sq, z['pen_sq.%d' % l]) < 1e-5
        sa, sc = model.full_sort_predict(inter)
        assert rel(sc, z['scores']) < 1e-4 and rel(sa, z['scores_att']) < 1e-4
        val, idx, rec = model.full_sort_topk(inter, c['k'], inter['item_id'])
        ok, nbad = O.topk_equal_modulo_ties(idx.cpu(), torch.from_numpy(z['topk_idx']), torch.from_numpy(z['scores']))
        assert ok, nbad
        want = torch.gather(torch.from_numpy(z['scores']), 1, idx.cpu())
        assert rel(val, want) < 1e-4
        pa, pc = model.predict(inter)
        assert rel(pa, z['predict_att']) < 1e-4 and rel(pc, z['predict_cal']) < 1e-4


def test_ssept_trainer_epoch_and_eval(A, tmp_path):
    """ACSSEPTTrainer: the adversarial two-loss step (routed double backward) + graphed full-sort evaluation, end to end"""
    cfg = O.default_cfg(n_layers=1)
    cfg.update(user_hidden_size=32, item_hidden_size=32)
    V = 200
    config = make_config(A, cfg, checkpoint_dir=str(tmp_path), epochs=1, train_batch_size=32, eval_batch_size=32, cuda_graph=True)
    config['model'] = 'ACSSEPT'
    torch.manual_seed(0)
    train_ds = A.data.SyntheticSequentialDataset(config, 32 * 3, V, seed=1)
    valid_ds = A.data.SyntheticSequentialDataset(config, 64, V, seed=2)
    model = A.ACSSEPT(config, train_ds).to('cuda')
    trainer = A.ACSSEPTTrainer(config, model)
    assert trainer.fused is None                      # the autograd path over the same kernels
    before_i = model.item_embedding.weight.detach().clone()
    before_u = model.user_embedding.weight.detach().clone()
    loader = A.data.TrainDataLoader(config, train_ds, shuffle=True)
    score, result = trainer.fit(loader, A.data.FullSortEvalDataLoader(config, valid_ds), verbose=False, saved=True)
    assert float((model.item_embedding.weight.detach() - before_i).abs().max()) > 0
    assert float((model.user_embedding.weight.detach() - before_u).abs().max()) > 0       # trained through the input concat
    assert all(np.isfinite(v) for v in result.values()) and 'hit@10' in result
    # the graphed evaluation and the eager one agree
    model.eval()
    batch = next(iter(A.data.FullSortEvalDataLoader(config, valid_ds)))
    rec_g = trainer.eval_batch(batch).cpu()
    trainer.use_graph = False
    rec_e = trainer.eval_batch(batch).cpu()
    assert torch.equal(rec_g, rec_e)


# ---- ACTiSASRec (SURVEY section 8 f-4): goldens from the real reference (tests/golden/make_golden.py: make_ti_case) ----
def build_ti(A, c, **extra):
    config = make_config(A, dict(c['cfg']), TIME_FIELD='timestamp', **extra)
    config['model'] = 'ACTiSASRec'
    model = A.ACTiSASRec(config, DS(c['V'])).to('cuda')
    model.load_state_dict({k: v.cuda() for k, v in c['params'].items()}, strict=True)      # reference state_dict loads unchanged
    model._debug_rand = {k: v.cuda() for k, v in c['rand'].d.items()}
    return config, model


def ti_inter(A, c):
    inter = inter_of(A, c)
    inter.interaction['timestamp_list'] = c['batch']['time'].cuda()
    return inter


@pytest.mark.parametrize('name', [n for n in TI if '_train' in n])
def test_ti_golden_train_losses_and_routed_grads(A, name):
    c = load_case(name)
    z = c['z']
    config, model = build_ti(A, c)
    model.train()
    l_att, l_cal = model.calculate_loss(ti_inter(A, c))
    assert abs(float(l_att) - float(z['loss_att'])) < 1e-4 * abs(float(z['loss_att']))
    assert abs(float(l_cal) - float(z['loss_cal'])) < 1e-4 * abs(float(z['loss_cal']))
    for n, p in model.named_parameters():
        p.requires_grad = not ('attack_key_transform' in n or 'attack_query_transform' in n)
    l_cal.backward(retain_graph=True)
    for n, p in model.named_parameters():
        p.requires_grad = ('attack_key_transform' in n or 'attack_query_transform' in n)
    l_att.backward()
    assert set(n for n, _ in model.named_parameters()) == set(c['grads'])
    for n, p in model.named_parameters():
        ref = c['grads'][n]
        got = p.grad.cpu() if p.grad is not None else torch.zeros_like(ref)
        scale = float(ref.abs().max())
        err = float((got - ref).abs().max())
        assert err <= 1e-3 * scale + 1e-8, (n, err, scale)


@pytest.mark.parametrize('name', [n for n in TI if '_eval' in n])
def test_ti_golden_eval(A, name):
    c = load_case(name)
    z = c['z']
    config, model = build_ti(A, c)
    model.eval()
    inter = ti_inter(A, c)
    with torch.no_grad():
        tm = model.get_time_matrix(inter['timestamp_list'])
        att, cal, masks = model.forward(inter['item_id_list'], inter['item_length'], tm)
        assert rel(att, z['out_att']) < 1e-4 and rel(cal, z['out_cal']) < 1e-4
        for l, m in enumerate(masks):
            assert rel(m.pen_sq, z['pen_sq.%d' % l]) < 1e-5
        sa, sc = model.full_sort_predict(inter)
        assert rel(sc, z['scores']) < 1e-4 and rel(sa, z['scores_att']) < 1e-4
        val, idx, rec = model.full_sort_topk(inter, c['k'], inter['item_id'])
        ok, nbad = O.topk_equal_modulo_ties(idx.cpu(), torch.from_numpy(z['topk_idx']), torch.from_numpy(z['scores']))
        assert ok, nbad
        pa, pc = model.predict(inter)
        assert rel(pa, z['predict_att']) < 1e-4 and rel(pc, z['predict_cal']) < 1e-4


def test_ti_trainer_epoch_and_eval(A, tmp_path):
    """ACTiSASRecTrainer: Philox dropout of the time-aware terms, routed double backward, graphed full-sort evaluation"""
    cfg = O.default_cfg(n_layers=2)
    cfg.update(time_span=64, TIME_FIELD='timestamp')
    V = 200
    config = make_config(A, cfg, checkpoint_dir=str(tmp_path), epochs=1, train_batch_size=32, eval_batch_size=32, cuda_graph=True)
    config['model'] = 'ACTiSASRec'
    torch.manual_seed(0)
    train_ds = A.data.SyntheticSequentialDataset(config, 32 * 3, V, seed=1)
    valid_ds = A.data.SyntheticSequentialDataset(config, 64, V, seed=2)
    model = A.ACTiSASRec(config, train_ds).to('cuda')
    trainer = A.ACTiSASRecTrainer(config, model)
    assert trainer.fused is None
    before = {n: p.detach().clone() for n, p in model.named_parameters()}
    score, result = trainer.fit(A.data.TrainDataLoader(config, train_ds, shuffle=True), A.data.FullSortEvalDataLoader(config, valid_ds),
                                verbose=False, saved=True)
    for n in ('item_embedding.weight', 'time_matrix_emb_K_embedding.weight', 'time_matrix_emb_V_embedding.weight',
              'absolute_pos_K_embedding.weight', 'absolute_pos_V_embedding.weight'):
        assert float((dict(model.named_parameters())[n].detach() - before[n]).abs().max()) > 0, n
    assert all(np.isfinite(v) for v in result.values()) and 'hit@10' in result
    model.eval()
    batch = next(iter(A.data.FullSortEvalDataLoader(config, valid_ds)))
    rec_g = trainer.eval_batch(batch).cpu()
    trainer.use_graph = False
    rec_e = trainer.eval_batch(batch).cpu()
    assert torch.equal(rec_g, rec_e)


@pytest.mark.parametrize('name', ['ACSSEPT', 'ACTiSASRec', 'AcBERT4Rec'])
def test_sibling_graphed_step_matches_eager(A, tmp_path, name):
    """sibling models with no host-side work in the step are captured in a CUDA graph by the trainer (forward + routed double
    backward + Adam through the autograd Functions); three graphed steps leave the same parameters as three eager ones"""
    cfg = O.default_cfg(n_layers=2)
    cfg.update(time_span=64, TIME_FIELD='timestamp', user_hidden_size=32, item_hidden_size=32, mask_ratio=0.2)
    V, B = 300, 32
    finals = []
    for use_graph in (True, False):
        import random
        random.seed(11)                        # AcBERT4Rec: the host-side masking stream (one reconstruct_train_data per step either way)
        config = make_config(A, cfg, checkpoint_dir=str(tmp_path), train_batch_size=B, eval_batch_size=B, cuda_graph=use_graph)
        config['model'] = name
        ds = A.data.SyntheticSequentialDataset(config, 3 * B, V, seed=4)
        torch.manual_seed(3)
        model = getattr(A, name)(config, ds).to('cuda')
        trainer = getattr(A, name + 'Trainer')(config, model)
        model.train()
        loader = A.data.TrainDataLoader(config, ds, shuffle=False)
        la, lc = trainer._train_epoch(loader, 0)
        assert (trainer._graph is not None) == use_graph
        assert np.isfinite(la) and np.isfinite(lc)
        finals.append((la, lc, {n: p.detach().clone() for n, p in model.named_parameters()}))
    (la_g, lc_g, pg), (la_e, lc_e, pe) = finals
    assert abs(la_g - la_e) < 1e-4 * abs(la_e) and abs(lc_g - lc_e) < 1e-4 * abs(lc_e)
    for n in pe:
        assert float((pg[n] - pe[n]).abs().max()) < 2e-5, n


@pytest.mark.parametrize('name', ['ACSSEPT', 'ACTiSASRec', 'ACSASRec'])
def test_direct_param_grads_equal_autograd_accumulation(A, tmp_path, name, monkeypatch):
    """the trainer's autograd step lets the backward kernels accumulate parameter gradients straight into the flat gradient buffer
    (ops.direct_param_grads) and skips gradients the routed double backward would drop; the flat gradient and the parameters after
    two steps equal those of plain autograd accumulation"""
    import contextlib
    cfg = O.default_cfg(n_layers=2)
    cfg.update(time_span=64, TIME_FIELD='timestamp', user_hidden_size=32, item_hidden_size=32)
    V, B = 300, 32
    finals = []
    ds = init = None
    for direct in (True, False):
        if not direct:
            monkeypatch.setattr(A.ops, 'direct_param_grads', contextlib.nullcontext)
            monkeypatch.setattr(A.ops, '_wants_grad', lambda t: t is not None)
        config = make_config(A, cfg, checkpoint_dir=str(tmp_path), train_batch_size=B, eval_batch_size=B, cuda_graph=False, fused_step=False)
        config['model'] = name
        # both runs start from the same batch and the same parameters, so the comparison is between the two gradient paths alone;
        # re-seeding the host initialisation does not promise bit-identical values, and a start difference survives Adam
        if ds is None:
            ds = A.data.SyntheticSequentialDataset(config, B, V, seed=4)
        torch.manual_seed(3)
        model = getattr(A, name)(config, ds).to('cuda')
        if init is None:
            init = {k: v.clone() for k, v in model.state_dict().items()}
        model.load_state_dict(init)
        trainer = getattr(A, name + 'Trainer')(config, model)
        assert trainer.fused is None
        model.train()
        batch = A.Interaction({k: v.cuda() for k, v in ds.inter_feat.interaction.items()})
        for _ in range(2):
            la, lc = trainer.train_step(batch)
        finals.append((float(la), float(lc), trainer.optimizer.flat_grad.clone(), trainer.optimizer.flat_param.clone()))
    (la1, lc1, g1, p1), (la0, lc0, g0, p0) = finals
    assert abs(la1 - la0) < 1e-5 * abs(la0) and abs(lc1 - lc0) < 1e-5 * abs(lc0)
    assert float((g1 - g0).abs().max()) <= 2e-5 * float(g0.abs().max())
    assert float((p1 - p0).abs().max()) < 5e-6
