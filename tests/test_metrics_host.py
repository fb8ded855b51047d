"""GAUC and the item-distribution metrics of the evaluator against the loop-based restatement of RecBole 1.0.1 (oracle/
metrics_oracle.py), on seeded integer score matrices with many ties.  The evaluator sees only what the evaluation kernels hand
over -- the positive's rank counts (items above, items tied), user_len, the top-k ids and the training item counts -- while the
oracle sorts the whole score matrix, as the reference does."""
import numpy as np
import pytest
import torch

from oracle import metrics_oracle as MO

NEW = ['gauc', 'itemcoverage', 'averagepopularity', 'giniindex', 'shannonentropy', 'tailpercentage']
OLD = ['hit', 'mrr', 'recall', 'ndcg', 'precision', 'map']


@pytest.fixture(scope='module')
def E():
    from ac_tsr_b200 import evaluator
    return evaluator


def make_case(seed, B=97, V=301, kmax=20, n_cand=None, span=6):
    """integer scores in [-span, span] (heavy ties), column 0 = -inf (trainer.py:942); n_cand: sampled evaluation, only the
    positive and n_cand - 1 other items are finite.  -> scores [B, V] float32, positives [B], top-k ids [B, kmax] (stable: lowest
    id first among ties), training counts [V] with zeros (items absent from the counter)"""
    g = np.random.default_rng(seed)
    s = g.integers(-span, span + 1, (B, V)).astype(np.float32)
    s[:, 0] = -np.inf
    pos = g.integers(1, V, B)
    s[0, :] = 0.0                                   # a user whose positive ties with every item
    s[0, 0] = -np.inf
    s[1, pos[1]] = span + 1                         # the positive as the best item
    s[2, pos[2]] = -span - 1                        # ... and as the worst
    if n_cand is not None:
        keep = np.zeros_like(s, dtype=bool)
        for b in range(B):
            keep[b, g.choice(np.arange(1, V), n_cand - 1, replace=False)] = True
            keep[b, pos[b]] = True
        keep[3, :] = False                          # a user whose only candidate is the positive: dropped from GAUC
        keep[3, pos[3]] = True
        s = np.where(keep, s, -np.inf).astype(np.float32)
    order = np.argsort(-s, axis=1, kind='stable')
    items = order[:, :kmax]
    counts = g.integers(0, 40, V)
    counts[g.random(V) < 0.3] = 0
    counts[0] = 0
    return s, pos, items, counts


def device_view(s, pos):
    """what the kernels hand over: (G, E) with the positive's own column excluded, user_len = finite scores"""
    sp = s[np.arange(s.shape[0]), pos][:, None]
    gt = (s > sp).sum(1)
    eq = (s == sp).sum(1) - 1
    return np.stack((gt, eq), 1).astype(np.int32), np.isfinite(s).sum(1).astype(np.int32)


def cfg(metrics, topk, tail=None, dp=4):
    c = {'metrics': metrics, 'topk': topk, 'metric_decimal_place': dp}
    if tail is not None:
        c['tail_ratio'] = tail
    return c


def run_both(E, s, pos, items, counts, metrics, topk, tail, dp=4):
    ev = E.Evaluator(cfg(metrics, topk, tail, dp))
    rec = np.concatenate(((items == pos[:, None]).astype(np.int32), np.ones((len(pos), 1), np.int32)), 1)
    c, ul = device_view(s, pos)
    got = ev.evaluate(rec, counts=c, user_len=ul, items=items.astype(np.int32), n_items=s.shape[1], item_counts=counts)
    counter = {int(i): int(n) for i, n in enumerate(counts) if n > 0}
    want = MO.evaluate([m for m in metrics if m in NEW], topk, torch.from_numpy(s), pos, items, s.shape[1], counter, tail, dp)
    return got, want


@pytest.mark.parametrize('seed', [0, 1, 2])
@pytest.mark.parametrize('topk', [[10], [1, 5, 20], [3, 7]])
@pytest.mark.parametrize('tail', [None, 0.1, 0.5, 3])
def test_new_metrics_equal_the_oracle(E, seed, topk, tail):
    s, pos, items, counts = make_case(seed, kmax=max(topk))
    got, want = run_both(E, s, pos, items, counts, NEW, topk, tail)
    assert list(got) == ['gauc'] + ['%s@%d' % (m, k) for m in NEW[1:] for k in topk]
    assert got == want


@pytest.mark.parametrize('dp', [2, 6])
def test_rounding_follows_metric_decimal_place(E, dp):
    s, pos, items, counts = make_case(5, kmax=10)
    got, want = run_both(E, s, pos, items, counts, NEW, [10], 0.5, dp)
    assert got == want
    assert all(round(v, dp) == v for v in got.values())


def test_tail_users_with_and_without_tail_items(E):
    """users whose lists hold no tail item, some, or only tail items"""
    s, pos, items, counts = make_case(7, kmax=10)
    tail = E.tail_items(counts, 0.5)
    tail_ids = np.nonzero(tail)[0]
    items[:10] = tail_ids[:10][None, :]                      # only tail items
    head = np.nonzero(~tail & (counts > 0))[0]
    items[10:20] = head[:10][None, :]                        # none
    got, want = run_both(E, s, pos, items, counts, ['tailpercentage', 'averagepopularity'], [1, 10], 0.5)
    assert got == want


@pytest.mark.parametrize('n_cand', [2, 11, 101])
def test_gauc_sampled_candidates(E, n_cand):
    s, pos, items, counts = make_case(11, n_cand=n_cand)
    got, want = run_both(E, s, pos, items, counts, ['gauc'], [10], None)
    assert got == want


def test_old_metrics_unchanged_and_order_kept(E):
    s, pos, items, counts = make_case(3, kmax=20)
    rec = np.concatenate(((items == pos[:, None]).astype(np.int32), np.ones((len(pos), 1), np.int32)), 1)
    old = E.Evaluator(cfg(OLD, [5, 20])).evaluate(rec)
    c, ul = device_view(s, pos)
    mixed = ['hit', 'gauc', 'mrr', 'itemcoverage', 'recall', 'ndcg', 'precision', 'map']
    res = E.Evaluator(cfg(mixed, [5, 20])).evaluate(rec, counts=c, user_len=ul, items=items, n_items=s.shape[1], item_counts=counts)
    assert {k: v for k, v in res.items() if k in old} == old
    assert [k.split('@')[0] for k in res][::1] == ['hit', 'hit', 'gauc', 'mrr', 'mrr', 'itemcoverage', 'itemcoverage', 'recall',
                                                  'recall', 'ndcg', 'ndcg', 'precision', 'precision', 'map', 'map']
    for m in OLD:                                  # the values themselves: the existing per-metric formulas
        avg = E.METRICS[m](rec[:, :-1].astype(bool), rec[:, -1].astype(np.int64)).mean(axis=0)
        assert old['%s@5' % m] == round(float(avg[4]), 4)


@pytest.mark.parametrize('m', ['AUC', 'LogLoss', 'MAE', 'RMSE', 'NoSuchMetric'])
def test_value_metrics_keep_raising(E, m):
    with pytest.raises(NotImplementedError):
        E.Evaluator(cfg(['Recall', m], [10]))


def test_trainer_config_errors_without_a_gpu():
    """item metrics under uni100 and popularity metrics without training counts are rejected before any kernel runs"""
    from ac_tsr_b200.trainer import ACSASRecTrainer

    class Loader(object):
        neg_sampler = object()
        neg_num = 100

        class dataset(object):
            item_num = 10

        def __iter__(self):
            raise AssertionError('no batch may be evaluated')

        def __len__(self):
            return 1

    t = ACSASRecTrainer.__new__(ACSASRecTrainer)
    t.model = torch.nn.Linear(1, 1)
    t.item_counts = None
    t.tot_item_num = None
    t.evaluator = __import__('ac_tsr_b200.evaluator', fromlist=['Evaluator']).Evaluator(cfg(['Recall', 'ItemCoverage'], [10]))
    with pytest.raises(NotImplementedError, match='sampled evaluation'):
        t.evaluate(Loader(), load_best_model=False)
    Loader.neg_sampler = None
    t.evaluator = __import__('ac_tsr_b200.evaluator', fromlist=['Evaluator']).Evaluator(cfg(['AveragePopularity'], [10]))
    with pytest.raises(ValueError, match='set_item_counts'):
        t.evaluate(Loader(), load_best_model=False)


def test_set_item_counts_is_the_training_bincount():
    from ac_tsr_b200.trainer import ACSASRecTrainer

    class DS(object):
        iid_field = 'item_id'
        item_num = 8
        inter_feat = {'item_id': torch.tensor([3, 1, 3, 7, 3, 1])}

    class Loader(object):
        dataset = DS()

    t = ACSASRecTrainer.__new__(ACSASRecTrainer)
    t.set_item_counts(Loader())
    assert t.item_counts.tolist() == [0, 2, 0, 3, 0, 0, 0, 1]
