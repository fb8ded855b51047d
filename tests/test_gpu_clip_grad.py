"""Gradient clipping by global norm on the device (`clip_grad_norm`, torch.nn.utils.clip_grad_norm_): the fp64 norm kernel
(acsr_grad_norm_partial) against torch.linalg.vector_norm, the clipped Adam (acsr_adam_step_clipped) against clip_grad_norm_ +
torch.optim.Adam, and the trainer: AC-SASRec's fused step and the sibling models' captured step with clipping on, against the
autograd step with torch's clip_grad_norm_, the fallbacks that keep torch's clip, and run_recbole end to end."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import acsr_oracle as O
from test_gpu_model import DS, make_config

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INF = float('inf')


@pytest.fixture(scope='module')
def A():
    import ac_tsr_b200 as pkg
    pkg.LIB.load()
    return pkg


def ref_partial(x, q):
    """sum |x|^q (max |x| for q = inf) in fp64, from torch.linalg.vector_norm"""
    n = torch.linalg.vector_norm(x.double(), q)
    return n if q == INF else n ** q


def rel_err(got, want):
    got, want = float(got), float(want)
    return abs(got - want) / max(abs(want), 1e-300)


# ---- the norm kernel ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize('n', [1, 3, 1000003, 64 * 10 ** 6 + 5])
@pytest.mark.parametrize('q', [1.0, 2.0, 3.5, INF])
def test_grad_norm_partial_matches_torch(A, n, q):
    g = torch.Generator(device='cuda').manual_seed(n % 1000)
    x = torch.randn(n, device='cuda', generator=g) * 1e-2
    got = A.ops.grad_norm_partial(x, q)
    assert got.dtype == torch.float64 and got.shape == (1,)
    assert rel_err(got, ref_partial(x, q)) <= 1e-6, (float(got), float(ref_partial(x, q)))
    # an unaligned view: scalar head and tail around the float4 body
    if n > 8:
        v = x[1:n - 2]
        assert rel_err(A.ops.grad_norm_partial(v, q), ref_partial(v, q)) <= 1e-6


@pytest.mark.parametrize('q', [2.0, INF])
def test_grad_norm_partial_walks_several_ranges_in_one_launch(A, q):
    x = torch.randn(3000017, device='cuda')
    ranges = [(0, 5), (7, 1000001), (1000001, 1000002), (2000003, 3000017), (9, 9)]
    got = A.ops.grad_norm_partial(x, q, ranges)
    parts = [x[b:e] for b, e in ranges if e > b]
    want = max(float(ref_partial(p, q)) for p in parts) if q == INF else sum(float(ref_partial(p, q)) for p in parts)
    assert rel_err(got, want) <= 1e-6
    # the same work pair serves consecutive launches (the last CTA resets the counter)
    work = A.ops.grad_norm_work(x.device)
    a = A.ops.grad_norm_partial(x, q, ranges[:2], work=work).clone()
    b = A.ops.grad_norm_partial(x, q, ranges[2:], work=work).clone()
    assert int(work[1].item()) == 0
    want_a = sum(float(ref_partial(x[s:e], q)) for s, e in ranges[:2]) if q != INF else max(float(ref_partial(x[s:e], q)) for s, e in ranges[:2])
    assert rel_err(a, want_a) <= 1e-6 and float(b) >= 0


def test_grad_norm_is_bit_identical_across_launches_and_graph_replay(A):
    x = torch.randn(64 * 10 ** 6 + 5, device='cuda')
    work = A.ops.grad_norm_work(x.device)
    out = torch.empty(1, dtype=torch.float64, device='cuda')
    first = A.ops.grad_norm_partial(x, 2.0, out=out, work=work).clone()
    second = A.ops.grad_norm_partial(x, 2.0, out=out, work=work).clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            A.ops.grad_norm_partial(x, 2.0, out=out, work=work)
    torch.cuda.current_stream().wait_stream(s)
    out.zero_()
    graph.replay()
    third = out.clone()
    graph.replay()
    assert torch.equal(first, second) and torch.equal(first, third) and torch.equal(first, out)


@pytest.mark.parametrize('q', [2.0, INF])
@pytest.mark.parametrize('bad', ['nan', 'inf'])
def test_non_finite_gradients_propagate_like_torch(A, q, bad):
    x = torch.randn(100003, device='cuda')
    x[77777] = float(bad)
    want_norm = torch.linalg.vector_norm(x, q)
    got = A.ops.grad_norm_partial(x, q)
    assert (torch.isnan(got) if bad == 'nan' else torch.isinf(got)).all(), float(got)
    assert bool(torch.isnan(want_norm)) == bool(torch.isnan(got).all())
    # the clipped step: the coefficient is NaN (NaN norm) or 0 (Inf norm) and the gradient is scaled by it, as in torch
    p = torch.randn_like(x)
    grad = x.clone()
    ref = torch.nn.Parameter(p.clone())
    ref.grad = x.clone()
    total_ref = torch.nn.utils.clip_grad_norm_([ref], 1.0, q, foreach=False)          # torch.linalg.vector_norm, as above
    total = A.ops.adam_step_clipped(p, grad, torch.zeros_like(p), torch.zeros_like(p), torch.zeros(1, dtype=torch.int64, device='cuda'),
                                    1e-3, got, q, 1.0)
    assert torch.equal(torch.isnan(total), torch.isnan(total_ref.view(1))) and torch.equal(torch.isinf(total), torch.isinf(total_ref.view(1)))
    assert torch.equal(torch.isnan(grad), torch.isnan(ref.grad))
    fin = torch.isfinite(ref.grad)
    assert torch.equal(grad[fin], ref.grad[fin])


def test_all_zero_gradient_keeps_coefficient_one(A):
    n = 4099
    x = torch.zeros(n, device='cuda')
    part = A.ops.grad_norm_partial(x, 2.0)
    assert float(part) == 0.0
    p = torch.randn(n, device='cuda')
    p0 = p.clone()
    total = A.ops.adam_step_clipped(p, x, torch.zeros_like(p), torch.zeros_like(p), torch.zeros(1, dtype=torch.int64, device='cuda'),
                                    1e-3, part, 2.0, 0.5)
    assert float(total) == 0.0 and torch.equal(x, torch.zeros_like(x)) and torch.equal(p, p0)


# ---- the clipped Adam ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize('q', [2.0, 1.0, 3.5, INF])
@pytest.mark.parametrize('side', ['clipped', 'unclipped'])
def test_clipped_adam_matches_clip_grad_norm_and_torch_adam(A, q, side):
    torch.manual_seed(0)
    sizes = [(300, 64), (64,), (7,), (64, 64)]
    ref = [torch.nn.Parameter(torch.randn(s, device='cuda') * 0.1) for s in sizes]
    adam = torch.optim.Adam(ref, lr=1e-3, weight_decay=0.01)
    n = sum(p.numel() for p in ref)
    flat_p = torch.cat([p.detach().reshape(-1) for p in ref]).contiguous()
    m, v = torch.zeros_like(flat_p), torch.zeros_like(flat_p)
    step = torch.zeros(1, dtype=torch.int64, device='cuda')
    for it in range(3):
        grads = [torch.randn(s, device='cuda') * (0.05 + 0.02 * it) for s in sizes]
        norm = float(torch.linalg.vector_norm(torch.cat([g.reshape(-1) for g in grads]).double(), q))
        max_norm = 0.5 * norm if side == 'clipped' else 2.0 * norm          # kept away from the norm on either side
        for p, g in zip(ref, grads):
            p.grad = g.clone()
        total_ref = torch.nn.utils.clip_grad_norm_(ref, max_norm, q)
        adam.step()
        flat_g = torch.cat([g.reshape(-1) for g in grads]).contiguous()
        part = A.ops.grad_norm_partial(flat_g, q)
        total = A.ops.adam_step_clipped(flat_p, flat_g, m, v, step, 1e-3, part, q, max_norm, weight_decay=0.01)
        assert rel_err(total, total_ref) <= 1e-6
        want_g = torch.cat([p.grad.reshape(-1) for p in ref])
        assert float((flat_g - want_g).abs().max()) <= 1e-6 * float(want_g.abs().max())
        if side == 'unclipped':
            assert torch.equal(flat_g, torch.cat([g.reshape(-1) for g in grads]))       # multiplied by exactly 1
        want_p = torch.cat([p.detach().reshape(-1) for p in ref])
        assert float((flat_p - want_p).abs().max()) <= 1e-6 * float(want_p.abs().max())
    assert int(step.item()) == 3 and flat_p.numel() == n


def test_clipped_adam_combines_partials_in_index_order(A):
    """a table shard's partial and the replicated part's, passed as separate partials, give the norm of the whole buffer"""
    x = torch.randn(100000, device='cuda')
    parts = torch.cat([A.ops.grad_norm_partial(x, 2.0, [(0, 30000), (70000, 100000)]), A.ops.grad_norm_partial(x, 2.0, [(30000, 50000)]),
                       A.ops.grad_norm_partial(x, 2.0, [(50000, 70000)])])
    p = torch.zeros_like(x)
    g = x.clone()
    total = A.ops.adam_step_clipped(p, g, torch.zeros_like(x), torch.zeros_like(x), torch.zeros(1, dtype=torch.int64, device='cuda'),
                                    1e-3, parts, 2.0, 1.0)
    assert rel_err(total, torch.linalg.vector_norm(x.double())) <= 1e-6


# ---- the trainer ----------------------------------------------------------------------------------------------------
def _acsasrec(A, cfg, V, params, noise, **extra):
    config = make_config(A, cfg, **extra)
    model = A.ACSASRec(config, DS(V)).to('cuda')
    model.load_state_dict({k: v.cuda() for k, v in params.items()})
    model._debug_rand = noise
    return config, model


def _batch(A, seq, ln, pos, neg=None):
    f = {'item_id_list': seq.cuda(), 'item_length': ln.cuda(), 'item_id': pos.cuda()}
    if neg is not None:
        f['neg_item_id'] = neg.cuda()
    return A.Interaction(f)


def _setup(loss_type):
    cfg = O.default_cfg(hidden_dropout_prob=0.0, attn_dropout_prob=0.0, loss_type=loss_type)
    V, B, L = 2003, 128, 50
    params = O.init_params(cfg, V, seed=3)
    seq, ln, pos = O.synth_batch(B, L, V, seed=6)
    neg = torch.randint(1, V, (B,), generator=torch.Generator().manual_seed(9)) if loss_type == 'BPR' else None
    g = torch.Generator().manual_seed(0)
    noise = {(l, 'noise'): torch.randn(B, cfg['n_heads'], L, L, generator=g).cuda() for l in range(cfg['n_layers'])}
    return cfg, V, params, (seq, ln, pos, neg), noise


@pytest.mark.parametrize('loss_type', ['CE', 'BPR'])
@pytest.mark.parametrize('norm_type', [2, 'inf'])
def test_fused_clipped_step_matches_autograd_and_clip_grad_norm(A, loss_type, norm_type):
    cfg, V, params, b, noise = _setup(loss_type)
    q = float(norm_type)
    # reference: the autograd step (two routed backward passes), torch's clip_grad_norm_, then Adam on the clipped gradient
    config, model = _acsasrec(A, cfg, V, params, noise, fused_step=False)
    trainer = A.ACSASRecTrainer(config, model)
    assert trainer.fused is None
    model.train()
    inter = _batch(A, *b)
    trainer.optimizer.zero_grad()
    la0, lc0 = model.calculate_loss(inter)
    trainer._route(attack=False); lc0.backward(retain_graph=True)
    trainer._route(attack=True); la0.backward()
    for p in model.parameters():
        p.requires_grad = True
    norm = float(torch.nn.utils.get_total_norm([p.grad for p in model.parameters()], q))
    max_norm = 0.5 * norm                              # coef ~ 0.5, away from 1
    total_ref = float(torch.nn.utils.clip_grad_norm_(model.parameters(), max_norm, q))
    trainer.optimizer.step()
    g_ref = {n: p.grad.detach().cpu().clone() for n, p in model.named_parameters()}
    p_ref = {n: p.detach().cpu().clone() for n, p in model.named_parameters()}
    # the fused step with clip_grad_norm on the device
    config, model = _acsasrec(A, cfg, V, params, noise, clip_grad_norm={'max_norm': max_norm, 'norm_type': norm_type})
    trainer = A.ACSASRecTrainer(config, model)
    assert trainer.fused is not None and not trainer.torch_clip and trainer.optimizer.clip == (max_norm, q)
    model.train()
    la1, lc1 = trainer.train_step(_batch(A, *b))
    assert abs(float(la1) - float(la0)) < 1e-4 * abs(float(la0)) and abs(float(lc1) - float(lc0)) < 1e-4 * abs(float(lc0))
    assert rel_err(trainer.optimizer.grad_norm, total_ref) < 1e-3
    for n, p in model.named_parameters():
        ref = g_ref[n]
        scale = float(ref.abs().max())
        assert float((p.grad.cpu() - ref).abs().max()) <= 1e-3 * scale + 1e-8, n          # p.grad holds the clipped gradient
        # Adam's first step moves every weight by ~lr * sign(g): compare where the gradient is not noise-level
        big = ref.abs() > 1e-2 * scale
        if bool(big.any()):
            assert float((p.detach().cpu() - p_ref[n])[big].abs().max()) < 2e-5, n


@pytest.mark.parametrize('loss_type', ['CE', 'BPR'])
@pytest.mark.parametrize('norm_type', [2, 'inf'])
def test_graphed_clipped_steps_equal_eager_steps(A, loss_type, norm_type):
    cfg, V, params, b, noise = _setup(loss_type)
    clip = {'max_norm': 0.5, 'norm_type': norm_type}
    finals = []
    for graph in (True, False):
        config, model = _acsasrec(A, cfg, V, params, noise, cuda_graph=graph, clip_grad_norm=clip)
        trainer = A.ACSASRecTrainer(config, model)
        assert trainer.fused is not None
        model.train()
        inter = A.Interaction({k: v.cpu() for k, v in _batch(A, *b).interaction.items()})
        for _ in range(2):
            la, lc = trainer.graphed_step(inter) if graph else trainer.train_step(inter.to('cuda'))
        if graph:
            assert trainer._graph is not None
        finals.append((float(la), float(lc), float(trainer.optimizer.grad_norm), trainer.optimizer.flat_param.clone()))
    (la_g, lc_g, n_g, p_g), (la_e, lc_e, n_e, p_e) = finals
    assert abs(la_g - la_e) < 1e-4 * abs(la_e) and abs(lc_g - lc_e) < 1e-4 * abs(lc_e)
    assert abs(n_g - n_e) <= 1e-4 * n_e
    assert float((p_g - p_e).abs().max()) < 1e-5


@pytest.mark.parametrize('name', ['AcBERT4Rec', 'ACSSEPT', 'ACTiSASRec'])
def test_sibling_graphed_clipped_step_matches_eager_torch_clip(A, tmp_path, name):
    """one captured step with the device clip == one eager step with torch's clip_grad_norm_ (an extra clip_grad_norm_ key,
    foreach, keeps torch's clip and rules out the graph)"""
    import random
    cfg = O.default_cfg(n_layers=2)
    cfg.update(time_span=64, TIME_FIELD='timestamp', user_hidden_size=32, item_hidden_size=32, mask_ratio=0.2)
    V, B = 300, 32
    finals = []
    init = None
    for device_clip in (True, False):
        clip = {'max_norm': 0.05, 'norm_type': 2} if device_clip else {'max_norm': 0.05, 'norm_type': 2, 'foreach': None}
        random.seed(11)
        config = make_config(A, cfg, checkpoint_dir=str(tmp_path), train_batch_size=B, eval_batch_size=B, cuda_graph=True,
                             clip_grad_norm=clip)
        config['model'] = name
        ds = A.data.SyntheticSequentialDataset(config, B, V, seed=4)
        torch.manual_seed(3)
        model = getattr(A, name)(config, ds).to('cuda')
        if init is None:
            init = {k: v.clone() for k, v in model.state_dict().items()}
        model.load_state_dict(init)
        trainer = getattr(A, name + 'Trainer')(config, model)
        assert trainer.torch_clip == (not device_clip)
        model.train()
        la, lc = trainer._train_epoch(A.data.TrainDataLoader(config, ds, shuffle=False), 0)
        assert (trainer._graph is not None) == device_clip
        assert np.isfinite(la) and np.isfinite(lc)
        finals.append((la, lc, trainer.optimizer.flat_grad.clone(), {n: p.detach().clone() for n, p in model.named_parameters()}))
    (la_g, lc_g, g_g, pg), (la_e, lc_e, g_e, pe) = finals
    assert abs(la_g - la_e) < 1e-4 * abs(la_e) and abs(lc_g - lc_e) < 1e-4 * abs(lc_e)
    assert float((g_g - g_e).abs().max()) <= 1e-4 * float(g_e.abs().max())          # both hold the clipped gradient
    for n in pe:
        assert float((pg[n] - pe[n]).abs().max()) < 2e-5, n


@pytest.mark.parametrize('extra', [dict(clip_grad_norm={'max_norm': 0.5, 'norm_type': 2, 'error_if_nonfinite': True}),
                                   dict(clip_grad_norm={'max_norm': 0.5}, learner='sgd'),
                                   dict(clip_grad_norm={'max_norm': 0.5, 'norm_type': 0})])
def test_settings_the_device_cannot_clip_keep_torch_clip_grad_norm(A, monkeypatch, extra):
    cfg, V, params, b, noise = _setup('CE')
    config, model = _acsasrec(A, cfg, V, params, noise, cuda_graph=True, **extra)
    trainer = A.ACSASRecTrainer(config, model)
    assert trainer.fused is None and trainer.torch_clip and getattr(trainer.optimizer, 'clip', None) is None
    calls = []
    real = torch.nn.utils.clip_grad_norm_

    def counting(*a, **k):
        calls.append(k)
        return real(*a, **k)
    monkeypatch.setattr(torch.nn.utils, 'clip_grad_norm_', counting)
    model.train()
    la, lc = trainer.train_step(_batch(A, *b))
    assert calls == [extra['clip_grad_norm']] and np.isfinite(float(lc))


def test_run_recbole_with_clip_grad_norm(A, tmp_path):
    cfg = tmp_path / 'clip.yaml'
    cfg.write_text('clip_grad_norm: {max_norm: 0.5, norm_type: 2}\nepochs: 1\ncheckpoint_dir: %s\n' % tmp_path)
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'run_recbole.py'), '--config_files',
                        os.path.join(ROOT, 'config', 'ml-100k.yaml') + ' ' + str(cfg)], cwd=ROOT, capture_output=True, text=True, timeout=900)
    log = r.stdout + r.stderr
    assert r.returncode == 0, log[-4000:]
    assert 'clip_grad_norm on the device (fused step)' in log, log[-4000:]
    assert 'test result' in log and 'nan' not in log.split('test result')[-1].lower(), log[-2000:]
