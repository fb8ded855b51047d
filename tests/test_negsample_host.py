"""Negative sampling, host side: `eval_args.mode` / `neg_sampling` parsing, the used-id sets and alias table ops.NegSampler
builds from the ml-100k splits, the oracle's sampled ranking on hand-built cases, and the C ABI of the two new kernels
(negsample.cu) without a GPU.  The reference is not available here, so nothing below is a golden from it: the used sets are
checked against a plain restatement of RecBole's get_used_ids (oracle.used_ids)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from oracle import acsr_oracle as O
from oracle import negsample_oracle as NO

import ac_tsr_b200 as A

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def ml100k_config(**extra):
    cd = dict(data_path=GOLD + '/', load_col={'inter': ['user_id', 'item_id', 'rating', 'timestamp']},
              eval_args={'split': {'LS': 'valid_and_test'}, 'group_by': 'user', 'order': 'TO', 'mode': 'full'},
              device=torch.device('cpu'), train_batch_size=256, eval_batch_size=256, seed=42, loss_type='CE')
    cd.update(extra)
    return A.Config(model='ACSASRec', dataset='ml-100k', config_dict=cd)


@pytest.fixture(scope='module')
def ml100k():
    config = ml100k_config()
    ds = A.create_dataset(config)
    return config, ds, ds.build()


def _split_ids(splits):
    return [(s.inter_feat['user_id'].numpy(), s.inter_feat['item_id'].numpy()) for s in splits]


# ---- parsing ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize('mode,want', [('full', ('full', 0)), (None, ('full', 0)), ('uni100', ('uniform', 100)),
                                       ('pop50', ('popularity', 50)), ('uni1', ('uniform', 1)), ('uni1000', ('uniform', 1000))])
def test_parse_eval_mode(mode, want):
    assert A.dataset.parse_eval_mode(mode) == want


@pytest.mark.parametrize('mode', ['labeled', 'uni', 'pop0', 'uni-5', 'full100', 'unix'])
def test_parse_eval_mode_rejects(mode):
    with pytest.raises(NotImplementedError, match=repr(mode).strip("'").replace('-', r'\-')):
        A.dataset.parse_eval_mode(mode)


def test_parse_neg_sampling():
    f = A.dataset.parse_neg_sampling
    assert f(ml100k_config(loss_type='BPR', neg_sampling={'uniform': 1})) == 'uniform'
    assert f(ml100k_config(loss_type='BPR', neg_sampling={'popularity': 1})) == 'popularity'
    assert f(ml100k_config(loss_type='BPR', neg_sampling=None)) is None
    assert f(ml100k_config(loss_type='CE', neg_sampling={'uniform': 1})) is None            # CE ignores it, as before
    assert f(ml100k_config(loss_type='CE', neg_sampling={'uniform': 5})) is None
    with pytest.raises(NotImplementedError, match='one negative'):
        f(ml100k_config(loss_type='BPR', neg_sampling={'uniform': 2}))
    with pytest.raises(ValueError):
        f(ml100k_config(loss_type='BPR', neg_sampling={'zipf': 1}))


def test_data_preparation_rejects_unsupported_modes(ml100k):
    config, ds, _ = ml100k
    config = ml100k_config(eval_args={'split': {'LS': 'valid_and_test'}, 'group_by': 'user', 'order': 'TO', 'mode': 'labeled'})
    with pytest.raises(NotImplementedError, match='labeled'):
        A.data_preparation(config, ds)
    config = ml100k_config(loss_type='BPR', neg_sampling={'uniform': 3})
    with pytest.raises(NotImplementedError, match='one negative'):
        A.data_preparation(config, ds)


def test_full_mode_loaders_unchanged(ml100k):
    """mode: full without neg_sampling: the same loader classes and the same batches as before the sampler existed"""
    config, ds, _ = ml100k
    tr, va, te = A.data_preparation(config, ds)
    # (by name: the package may be imported under both of its module names by other tests)
    assert [type(x).__name__ for x in (tr, va, te)] == ['TrainDataLoader', 'FullSortEvalDataLoader', 'FullSortEvalDataLoader']
    assert getattr(tr, 'neg_sampler', None) is None and not hasattr(va, 'neg_sampler')
    fields = ['item_id_list', 'item_length', 'item_id']
    assert tr._packed.fields == fields and va._packed.fields == fields
    inter, hist, pu, pi = next(iter(va))
    assert hist is None and torch.equal(pu, torch.arange(len(inter))) and torch.equal(pi, inter['item_id'])
    assert sorted(inter.interaction.keys()) == sorted(fields)
    va.pr = 0


def test_sampled_mode_loaders(ml100k):
    config, ds, _ = ml100k
    config = ml100k_config(eval_args={'split': {'LS': 'valid_and_test'}, 'group_by': 'user', 'order': 'TO', 'mode': 'pop100'})
    tr, va, te = A.data_preparation(config, ds)
    assert type(va).__name__ == 'NegSampleEvalDataLoader' and va.neg_num == 100 and va.neg_sampler.distribution == 'popularity'
    assert te.neg_sampler.rng_stream != va.neg_sampler.rng_stream
    assert getattr(tr, 'neg_sampler', None) is None                 # CE training: no training sampler
    inter, hist, pu, pi = next(iter(va))
    va.pr = 0
    assert hist is None and torch.equal(pi, inter['item_id']) and 'user_id' in inter
    config = ml100k_config(loss_type='BPR', neg_sampling={'uniform': 1})
    tr, va, _ = A.data_preparation(config, ds)
    assert type(va).__name__ == 'FullSortEvalDataLoader'
    assert tr.neg_sampler.distribution == 'uniform' and 'user_id' in tr._packed.fields
    batch = next(iter(tr))
    tr.pr = 0
    assert 'user_id' in batch and 'neg_item_id' not in batch


# ---- used sets / alias table -----------------------------------------------------------------------------
@pytest.mark.parametrize('phase', [0, 1, 2])
def test_used_sets_match_recbole_get_used_ids(ml100k, phase):
    config, ds, splits = ml100k
    samplers = A.dataset.build_neg_samplers(config, splits, 'uniform', 'uniform')
    s = samplers[phase]
    want = NO.used_ids(_split_ids(splits), ds.user_num, phase)
    off, items = s.used_offsets, s.used_items
    assert len(off) == ds.user_num + 1 and off[0] == 0 and off[-1] == len(items)
    for u in range(ds.user_num):
        row = items[off[u]:off[u + 1]]
        assert np.all(np.diff(row) > 0), u
        assert set(row.tolist()) == want[u], u
    # a history's first item is only ever inside item_id_list, never a target: it stays drawable
    tr = splits[0].inter_feat
    first = tr['item_length'].numpy() == 1
    n_checked = 0
    for u, it in zip(tr['user_id'].numpy()[first], tr['item_id_list'].numpy()[first, 0]):
        if it not in want[u]:
            row = items[off[u]:off[u + 1]]
            assert it not in row
            n_checked += 1
    assert n_checked > 0


def test_alias_table_probabilities(ml100k):
    config, ds, splits = ml100k
    s = A.dataset.build_neg_samplers(config, splits, None, 'popularity')[1]
    want = NO.popularity_probs(_split_ids(splits), ds.item_num)
    got = NO.alias_probs(*s.alias)
    assert want[0] == 0.0 and np.abs(got - want).max() <= 1e-6
    for counts in (np.array([0, 1, 1, 1, 1.0]), np.array([0, 100, 1, 0, 3.0]), np.random.default_rng(0).zipf(1.5, 5000).astype(float)):
        assert np.abs(NO.alias_probs(*A.ops.alias_table(counts)) - counts / counts.sum()).max() <= 1e-6


def test_popularity_fallback_share_on_ml100k(ml100k):
    """how often popN / popularity negatives leave the alias draw for the uniform-complement fallback: with probability f^16 per
    negative, f = the popularity mass of the user's used set.  On ml-100k that is at most 0.33 % (the heaviest user, f = 0.70)
    and 1e-5 on average, so popN metrics are those of the exact restricted popularity distribution to well below 1e-4"""
    config, ds, splits = ml100k
    for s in A.dataset.build_neg_samplers(config, splits, 'popularity', 'popularity'):
        p = s.counts / s.counts.sum()
        f = np.add.reduceat(np.r_[p[s.used_items], 0.0], s.used_offsets[:-1]) * (np.diff(s.used_offsets) > 0)
        fb = f ** 16
        assert fb.max() < 5e-3 and fb[1:].mean() < 2e-5


def test_alias_table_shared_between_phases(ml100k):
    config, ds, splits = ml100k
    ss = A.dataset.build_neg_samplers(config, splits, 'popularity', 'popularity')
    assert ss[0].alias is ss[1].alias is ss[2].alias


def test_loaders_reject_user_ids_outside_the_sampler():
    off, items = A.ops.used_item_csr([1, 2], [1, 2], 3, 10)
    s = A.ops.NegSampler('uniform', off, items, 10, seed=0)
    s.check_users(np.array([0, 1, 2]))
    with pytest.raises(ValueError, match='user ids'):
        s.check_users(np.array([1, 3]))


def test_sampler_rejects_a_user_without_negatives():
    off, items = A.ops.used_item_csr([1, 1, 1], [1, 2, 3], 2, 4)
    with pytest.raises(ValueError, match='every item'):
        A.ops.NegSampler('uniform', off, items, 4, seed=0)


# ---- oracle sampled ranking on hand-built cases -------------------------------------------------------------
def test_oracle_sampled_ranking_duplicates_and_ties():
    V, kmax = 10, 3
    # row 0: the positive (item 5) beaten by item 3 twice (a duplicate): rank 1, not 2
    # row 1: beaten by 3 distinct items: rank 3 = kmax -> no hit
    # row 2: a negative ties with the positive exactly: either rank is right, the bounds say [0, 1]
    cand = torch.tensor([[5, 3, 3, 7], [5, 1, 2, 4], [5, 6, 8, 9]])
    scores = torch.tensor([[1.0, 2.0, 2.0, 0.5], [0.0, 1.0, 2.0, 3.0], [1.0, 1.0, 0.0, -1.0]])
    flags, idx, full = NO.sampled_topk(scores, cand, V, kmax)
    assert flags[0].tolist() == [0, 1, 0] and flags[1].tolist() == [0, 0, 0]
    lo, hi = NO.sampled_rank_bounds(full, cand[:, 0])
    assert lo.tolist() == [1, 3, 0] and hi.tolist() == [1, 3, 1]
    assert NO.flags_rank(flags, kmax).tolist()[:2] == [1, 3]
    # item 0 never appears as a negative, and the -inf padding of the scattered matrix ranks below every candidate
    assert torch.isinf(full[0, 0]) and NO.flags_rank(torch.tensor([[0, 0, 1, 1]]), 3).tolist() == [2]


# ---- the C ABI of negsample.cu ----------------------------------------------------------------------------------
def test_negsample_cross_compiles_for_sm100a(tmp_path):
    from importlib import import_module
    b = import_module('ac-tsr_b200.build')
    src = os.path.join(b.CSRC, 'negsample.cu')
    r = subprocess.run([b._nvcc()] + b.NVCC_FLAGS + ['-c', src, '-o', str(tmp_path / 'negsample.o')], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert 'spill' not in r.stderr or ' 0 bytes spill stores' in r.stderr


def test_negsample_symbols_exported_and_reject_bad_arguments():
    import __graft_entry__ as g
    g.build()
    dll = ctypes.CDLL(A._lib.LIB_PATH)
    for name in ('acsr_neg_sample', 'acsr_candidate_rank', 'acsr_candidate_rank_max_candidates'):
        assert hasattr(dll, name) and name in A._lib.parse_header()
    assert A.LIB.query('acsr_candidate_rank_max_candidates') >= 1001
    with pytest.raises(A.AcsrError, match='NULL'):
        A.LIB.call('acsr_neg_sample', None, None, None, None, 0, 4, 1, None, None, 1, 10, None, None, None, 0, None, 1, None)
    fake = 1 << 20                                                     # never dereferenced: every check below fails first
    with pytest.raises(A.AcsrError, match='perm and cursor'):
        A.LIB.call('acsr_neg_sample', fake, None, fake, None, 8, 4, 1, fake, fake, 1, 10, None, None, fake, 0, fake, 1, None)
    with pytest.raises(A.AcsrError, match='bad sizes'):
        A.LIB.call('acsr_neg_sample', fake, None, None, None, 0, 4, 2, fake, fake, 1, 10, None, None, fake, 0, fake, 1, None)
    with pytest.raises(A.AcsrError, match='NULL'):
        A.LIB.call('acsr_candidate_rank', None, None, 10, 64, None, 4, 101, 10, None, None, None)
    with pytest.raises(A.AcsrError, match='at most 8191 negatives'):
        A.LIB.call('acsr_candidate_rank', fake, fake, 10, 64, fake, 4, 8193, 10, fake, None, None)
    with pytest.raises(A.AcsrError, match='1..1024'):
        A.LIB.call('acsr_candidate_rank', fake, fake, 10, 64, fake, 4, 101, 1025, fake, None, None)
    with pytest.raises(A.AcsrError, match='at most 1024'):
        A.LIB.call('acsr_candidate_rank', fake, fake, 10, 1028, fake, 4, 101, 10, fake, None, None)
    with pytest.raises(A.AcsrError, match='multiple of 4'):
        A.LIB.call('acsr_candidate_rank', fake, fake, 10, 30, fake, 4, 101, 10, fake, None, None)
    assert A._lib.ALGO_BYTES['acsr_candidate_rank']((0, 0, 10, 64, 0, 256, 101, 50, 0, None, None)) == \
        4 * 256 * 64 + 256 * 101 * (8 + 256) + 4 * 256 * 51


def test_sampler_and_rank_need_cuda_tensors():
    off, items = A.ops.used_item_csr([1, 1], [1, 2], 2, 10)
    s = A.ops.NegSampler('uniform', off, items, 10, seed=0)
    with pytest.raises(Exception):
        s.draw(torch.tensor([1]), 4)
    with pytest.raises(RuntimeError, match='disagree'):             # AcsrError, under either of the package's module names
        A.ops.candidate_rank(torch.zeros(2, 8), torch.zeros(10, 4), torch.zeros(2, 5, dtype=torch.int64), 3)
    with pytest.raises(RuntimeError, match='disagree'):
        A.ops.candidate_rank(torch.zeros(2, 8), torch.zeros(10, 8), torch.zeros(3, 5, dtype=torch.int64), 3)
    with pytest.raises(RuntimeError, match='CUDA'):
        A.ops.candidate_rank(torch.zeros(2, 8), torch.zeros(10, 8), torch.zeros(2, 5, dtype=torch.int64), 3)
