"""Atomic-file sequential dataset: the caller side of the hot path (SURVEY §8 f-1).

Rebuilds, for sequential models, what the reference does between a `<dataset>.inter` file and the three data loaders:

  recbole/data/dataset/dataset.py:405-452    typed-header atomic file (`field:type`, tab separated), `load_col`
  dataset.py:160-178, 624-668, 803-821       drop rows without user / item, `rm_dup_inter`, `val_interval`
  dataset.py:670-760                         k-core filtering by `user_inter_num_interval` / `item_inter_num_interval`
  dataset.py:920-974                         id remapping: `pandas.factorize` order of first appearance, id 0 = [PAD]
  dataset.py:1296-1318                       token -> int64, float -> float32 tensors
  sequential_dataset.py:73-135               augmentation: every prefix of a user's (time-sorted) history is one row
  dataset.py:1467-1510, 1398-1450            `eval_args`: order TO (stable sort by the target's time), split LS leave-one-out
  recbole/data/utils.py:96-150               data_preparation -> TrainDataLoader, FullSortEvalDataLoader (valid, test)

All of it is vectorised numpy (the reference loops in Python over interactions); results are bit-identical to the reference's
pipeline (tests/test_dataset_pipeline.py compares every tensor on ml-100k).  Only the fields the model reads are materialised
(`item_id_list`, `item_length`, `item_id`, `user_id`; the reference also builds `rating_list` / `timestamp_list`, which nothing
consumes -- SURVEY a19).  Out of scope here: user / item side-feature files, knowledge graphs, `RS` splits.  Negative sampling
(`neg_sampling` for BPR, `eval_args.mode: uniN / popN`) is drawn on the device (ops.NegSampler); this module builds its used sets.
"""
import copy
import gzip
import math
import os

import numpy as np
import torch

from .compat import Interaction, cfg_get


# ---------------------------------------------------------------------------------------------
# atomic files
# ---------------------------------------------------------------------------------------------
def read_atomic_file(path, load_col=None, field_separator='\t'):
    """-> ({field: np.ndarray (object for token, float64 for float)}, {field: type}); `path` may be gzip-compressed."""
    opener = gzip.open if path.endswith('.gz') else open
    with opener(path, 'rt', encoding='utf-8') as fh:
        header = fh.readline().rstrip('\n').split(field_separator)
        fields, ftypes = [], []
        for h in header:
            name, typ = h.split(':')
            if typ not in ('token', 'float', 'token_seq', 'float_seq'):
                raise ValueError('Type %s from field %s is not supported.' % (typ, name))          # dataset.py:421-423
            fields.append(name)
            ftypes.append(typ)
        keep = [i for i, f in enumerate(fields) if load_col is None or f in load_col]
        for i in keep:
            if ftypes[i] not in ('token', 'float'):
                raise NotImplementedError('sequence-typed columns of an .inter file are out of scope (field %s)' % fields[i])
        cols = [[] for _ in keep]
        for line in fh:
            parts = line.rstrip('\n').split(field_separator)
            if len(parts) < len(fields):
                parts += [''] * (len(fields) - len(parts))
            for c, i in zip(cols, keep):
                c.append(parts[i])
    data, types = {}, {}
    for c, i in zip(cols, keep):
        if ftypes[i] == 'float':
            data[fields[i]] = np.array([float(x) if x != '' else np.nan for x in c], dtype=np.float64)
        else:
            data[fields[i]] = np.array(c, dtype=object)
        types[fields[i]] = ftypes[i]
    return data, types


def _parse_intervals(s):
    """dataset.py:760-786: "[5,inf)" or "(0,1];[3,4)" -> [(left_bracket, lo, hi, right_bracket)]"""
    if s is None:
        return None
    out = []
    for part in str(s).split(';'):
        part = part.strip()
        lb, rb = part[0], part[-1]
        lo, hi = part[1:-1].split(',')
        out.append((lb, float(lo), float(hi), rb))
    return out


def _within(num, intervals):
    num = np.asarray(num, dtype=np.float64)
    res = np.zeros(num.shape, dtype=bool)
    for lb, lo, hi, rb in intervals:
        t = (num >= lo) if lb == '[' else (num > lo)
        t &= (num <= hi) if rb == ']' else (num < hi)
        res |= t
    return res


def _factorize(tokens):
    """order-of-first-appearance codes (pandas.factorize) -> (codes int64, uniques)"""
    uniq, first, inv = np.unique(tokens, return_index=True, return_inverse=True)
    order = np.argsort(first, kind='stable')
    rank = np.empty_like(order)
    rank[order] = np.arange(len(order))
    return rank[inv].astype(np.int64), uniq[order]


# ---------------------------------------------------------------------------------------------
class SequentialDataset(object):
    """`SequentialDataset(config)` -- same constructor contract as the reference's (create_dataset, data/utils.py:30-62)."""

    def __init__(self, config, inter_file=None):
        self.config = config
        self.dataset_name = config['dataset']
        self.uid_field = config['USER_ID_FIELD']
        self.iid_field = config['ITEM_ID_FIELD']
        self.time_field = config['TIME_FIELD']
        self.max_item_list_len = config['MAX_ITEM_LIST_LENGTH']
        self.item_list_length_field = config['ITEM_LIST_LENGTH_FIELD']
        self.item_id_list_field = self.iid_field + config['LIST_SUFFIX']
        self.field2id_token, self.field2token_id = {}, {}
        self.inter_feat = None
        if inter_file is None:
            base = os.path.join(config['data_path'], '%s.inter' % self.dataset_name)
            inter_file = base if os.path.isfile(base) else base + '.gz'
        if not os.path.isfile(inter_file):
            raise ValueError('File %s not exist.' % inter_file)                                       # dataset.py:337-338
        self._from_scratch(inter_file)

    # -- loading + filtering + remapping ------------------------------------------------------------
    def _from_scratch(self, inter_file):
        c = self.config
        load_col = (c['load_col'] or {}).get('inter') if c['load_col'] is not None else None
        data, types = read_atomic_file(inter_file, load_col, c['field_separator'] or '\t')
        for need in (self.uid_field, self.iid_field, self.time_field):
            if need not in data:
                raise ValueError('%s must be loaded for a sequential dataset (load_col.inter)' % need)
        n = len(data[self.uid_field])
        keep = np.ones(n, dtype=bool)
        for f in (self.uid_field, self.iid_field):                     # _filter_nan_user_or_item
            keep &= np.array([x != '' for x in data[f]], dtype=bool)
        data = {k: v[keep] for k, v in data.items()}
        data = self._remove_duplication(data)
        data = self._filter_by_field_value(data, types)
        data = self._filter_by_inter_num(data)
        # ids: 1.. in order of first appearance, 0 = [PAD]
        for f in (self.uid_field, self.iid_field):
            codes, uniq = _factorize(data[f])
            data[f] = codes + 1
            self.field2id_token[f] = np.array(['[PAD]'] + list(uniq), dtype=object)
            self.field2token_id[f] = {t: i for i, t in enumerate(self.field2id_token[f])}
        self.user_num = len(self.field2id_token[self.uid_field])
        self.item_num = len(self.field2id_token[self.iid_field])
        self.inter_num_raw = len(data[self.uid_field])
        self._raw = {self.uid_field: data[self.uid_field].astype(np.int64), self.iid_field: data[self.iid_field].astype(np.int64),
                     self.time_field: data[self.time_field].astype(np.float32)}     # float fields become float32 tensors
        self._augment()

    def _remove_duplication(self, data):
        keep = self.config['rm_dup_inter']
        if keep is None:
            return data
        # DataFrame.sort_values(by=[time]) (dataset.py:658): pandas' default kind is numpy's quicksort, which is NOT stable, and the
        # later sorts are, so the order it leaves equal timestamps in survives into the id numbering and the sequences.  The
        # same numpy call on the same float64 column reproduces it (same numpy build / CPU dispatch as the reference run).
        order = np.argsort(data[self.time_field], kind='quicksort')
        data = {k: v[order] for k, v in data.items()}
        pair = np.array(['%s\x00%s' % (u, i) for u, i in zip(data[self.uid_field], data[self.iid_field])], dtype=object)
        if keep == 'first':
            _, idx = np.unique(pair, return_index=True)
        elif keep == 'last':
            _, idx = np.unique(pair[::-1], return_index=True)
            idx = len(pair) - 1 - idx
        else:
            raise ValueError('rm_dup_inter must be first / last / None')
        idx = np.sort(idx)
        return {k: v[idx] for k, v in data.items()}

    def _filter_by_field_value(self, data, types):
        vi = self.config['val_interval'] or {}
        for field, interval in vi.items():
            if field not in data:
                raise ValueError('Field [%s] not defined in dataset.' % field)
            if types[field] == 'float':
                keep = _within(data[field], _parse_intervals(interval))
            else:
                keep = np.isin(data[field], list(interval))
            data = {k: v[keep] for k, v in data.items()}
        return data

    def _filter_by_inter_num(self, data):
        ui = _parse_intervals(self.config['user_inter_num_interval'])
        ii = _parse_intervals(self.config['item_inter_num_interval'])
        if ui is None and ii is None:
            return data
        ucode, _ = _factorize(data[self.uid_field])
        icode, _ = _factorize(data[self.iid_field])
        alive = np.ones(len(ucode), dtype=bool)
        while True:                                                    # k-core: repeat until nothing is dropped
            ucnt = np.bincount(ucode[alive], minlength=ucode.max() + 1 if len(ucode) else 0)
            icnt = np.bincount(icode[alive], minlength=icode.max() + 1 if len(icode) else 0)
            bad_u = ~_within(ucnt, ui) if ui is not None else np.zeros(len(ucnt), dtype=bool)
            bad_i = ~_within(icnt, ii) if ii is not None else np.zeros(len(icnt), dtype=bool)
            bad_u &= ucnt > 0                                          # ids without interactions left are not "illegal" any more
            bad_i &= icnt > 0
            drop = alive & (bad_u[ucode] | bad_i[icode])
            if not drop.any():
                break
            alive &= ~drop
        return {k: v[alive] for k, v in data.items()}

    # -- augmentation (sequential_dataset.py:73-135) --------------------------------------------------
    def _augment(self):
        L = self.max_item_list_len
        uid, iid, t = self._raw[self.uid_field], self._raw[self.iid_field], self._raw[self.time_field]
        order = np.argsort(t, kind='stable')
        order = order[np.argsort(uid[order], kind='stable')]           # Interaction.sort(by=[uid, time]): stable, last key first
        uid, iid, t = uid[order], iid[order], t[order]
        n = len(uid)
        idx = np.arange(n)
        is_first = np.ones(n, dtype=bool)
        is_first[1:] = uid[1:] != uid[:-1]
        start_of_user = np.maximum.accumulate(np.where(is_first, idx, 0))
        pos = idx - start_of_user                                      # items of this user before row i
        tgt = idx[~is_first]
        length = np.minimum(pos[tgt], L)
        seq_start = tgt - length
        cols = np.arange(L)
        gather = seq_start[:, None] + cols[None, :]
        valid = cols[None, :] < length[:, None]
        item_list = np.where(valid, iid[np.minimum(gather, n - 1)], 0)
        feat = {
            self.uid_field: torch.from_numpy(uid[tgt].copy()),
            self.iid_field: torch.from_numpy(iid[tgt].copy()),
            self.time_field: torch.from_numpy(t[tgt].copy()),
            self.item_list_length_field: torch.from_numpy(length.astype(np.int64)),
            self.item_id_list_field: torch.from_numpy(item_list.astype(np.int64)),
        }
        if str(self.config.get('model', '')) == 'ACTiSASRec':       # the one model that reads timestamp_list (actisasrec.py:35, 177)
            time_list = np.where(valid, t[np.minimum(gather, n - 1)], 0).astype(np.float32)
            feat[self.time_field + self.config['LIST_SUFFIX']] = torch.from_numpy(time_list)
        self.inter_feat = Interaction(feat)

    # -- API the model / trainer / loaders use ---------------------------------------------------------
    def num(self, field):
        if field in (self.iid_field, self.item_id_list_field):
            return self.item_num
        if field == self.uid_field:
            return self.user_num
        raise ValueError('field [%s] not defined in dataset' % field)

    def __len__(self):
        return len(self.inter_feat)

    def copy(self, new_inter_feat):
        nxt = copy.copy(self)
        nxt.inter_feat = new_inter_feat
        return nxt

    def __str__(self):
        return '%s\nThe number of users: %d\nThe number of items: %d\nThe number of inters: %d\nRemain Fields: %s' % (
            self.dataset_name, self.user_num, self.item_num, len(self), list(self.inter_feat.columns))

    # -- ordering + splitting (dataset.py:1467-1510) ---------------------------------------------------
    def build(self):
        ea = self.config['eval_args'] or {}
        if ea.get('order') != 'TO':
            raise ValueError('The ordering args for sequential recommendation has to be \'TO\'')       # sequential_dataset.py:211-213
        split = ea.get('split') or {}
        if list(split.keys()) != ['LS']:
            raise NotImplementedError('The splitting_method %s has not been implemented (LS only).' % list(split.keys()))
        mode = split['LS']
        feat = self.inter_feat
        order = np.argsort(feat[self.time_field].numpy(), kind='stable')
        uid = feat[self.uid_field].numpy()[order]
        n = len(uid)
        # leave-one-out per user, users in order of first appearance, rows in time order (dataset.py:1398-1450)
        ucode, _ = _factorize(uid)
        by_user = np.argsort(ucode, kind='stable')                     # rows grouped by user, time order kept inside a group
        cnt = np.bincount(ucode)
        ends = np.cumsum(cnt)
        rank_from_end = np.empty(n, dtype=np.int64)
        rank_from_end[by_user] = np.repeat(ends, cnt) - 1 - np.arange(n)
        tot = cnt[ucode]
        leave = {'valid_and_test': 2, 'valid_only': 1, 'test_only': 1}.get(mode)
        if leave is None:
            raise NotImplementedError('The leave_one_mode [%s] has not been implemented.' % mode)
        legal = np.minimum(leave, tot - 1)
        part = np.zeros(n, dtype=np.int64)                             # 0 train, 1.. = left-out parts counted from the END
        held = rank_from_end < legal
        part[held] = leave - rank_from_end[held]
        # rows of a part are collected user by user (in order of first appearance), not in global time order
        sel = [by_user[part[by_user] == k] for k in range(leave + 1)]
        if mode == 'valid_only':
            sel.append(np.zeros(0, dtype=np.int64))
        elif mode == 'test_only':
            sel = [sel[0], np.zeros(0, dtype=np.int64), sel[1]]
        out = []
        for s in sel:
            rows = torch.from_numpy(order[s])
            out.append(self.copy(Interaction({k: v[rows] for k, v in feat.interaction.items() if k != self.time_field})))
        return out


# ---------------------------------------------------------------------------------------------
def create_dataset(config):
    """data/utils.py:30-62 for MODEL_TYPE sequential"""
    return SequentialDataset(config)


def device_resident_training(config):
    """HBM-resident training data (data.DeviceTrainDataLoader) is AC-SASRec's: its fused step gathers the batch inside the captured
    graph.  The sibling models read more fields (user id, time stamps) or prepare the batch on the host (AcBERT4Rec's python
    masking) and take pinned host batches from TrainDataLoader."""
    dev = config['device']
    return (getattr(dev, 'type', str(dev)) == 'cuda' and bool(config.get('device_resident_data', True))
            and str(config.get('model', 'ACSASRec')) == 'ACSASRec')


def parse_eval_mode(mode):
    """eval_args.mode (config/configurator.py, data/utils.py:96-150) -> ('full', 0) | ('uniform', N) | ('popularity', N)"""
    m = str('full' if mode is None else mode)
    if m == 'full':
        return 'full', 0
    for prefix, dist in (('uni', 'uniform'), ('pop', 'popularity')):
        if m.startswith(prefix) and m[len(prefix):].isdigit() and int(m[len(prefix):]) > 0:
            return dist, int(m[len(prefix):])
    raise NotImplementedError('eval_args.mode %r: only full, uniN and popN evaluation are implemented' % m)


def parse_neg_sampling(config):
    """`neg_sampling` -> 'uniform' | 'popularity' | None.  Only loss_type BPR reads it (with CE it is ignored, as in the reference's
    sequential models); one negative per row, since RecBole repeats the batch rows for more."""
    ns = config['neg_sampling']
    if not ns or str(cfg_get(config, 'loss_type', 'CE')) != 'BPR':
        return None
    if not isinstance(ns, dict) or len(ns) != 1:
        raise ValueError('neg_sampling must be one of {uniform: 1} / {popularity: 1} (got %r)' % (ns,))
    (dist, num), = ns.items()
    if dist not in ('uniform', 'popularity'):
        raise ValueError('neg_sampling distribution %r: must be uniform or popularity' % (dist,))
    if int(num) != 1:
        raise NotImplementedError('neg_sampling {%s: %s}: only one negative per training row is implemented' % (dist, num))
    return dist


def build_neg_samplers(config, splits, train_dist, eval_dist):
    """-> (train, valid, test) ops.NegSampler | None.  Used ids of a phase: the targets of the user's rows in the splits up to
    and including it (sampler.py get_used_ids; a history's first item is never a target and stays drawable); popularity: the
    item counts over the targets of all three splits."""
    from .ops import NegSampler, alias_table, used_item_csr
    ds = splits[0]
    uf, itf = ds.uid_field, ds.iid_field
    n_users, n_items = ds.user_num, ds.item_num
    uids = [s.inter_feat[uf].numpy() for s in splits]
    iids = [s.inter_feat[itf].numpy() for s in splits]
    counts = np.bincount(np.concatenate(iids), minlength=n_items).astype(np.float64)
    seed = int(config['seed'] if config['seed'] is not None else 0)
    alias = alias_table(counts) if 'popularity' in (train_dist, eval_dist) else None       # built once, shared by the phases
    out = []
    for phase, dist in enumerate((train_dist, eval_dist, eval_dist)):
        if dist is None:
            out.append(None)
            continue
        off, items = used_item_csr(np.concatenate(uids[:phase + 1]), np.concatenate(iids[:phase + 1]), n_users, n_items)
        out.append(NegSampler(dist, off, items, n_items, seed, phase=phase, counts=counts, alias=alias))
    return out


def data_preparation(config, dataset):
    """data/utils.py:96-150 -> (train_data, valid_data, test_data)"""
    from .data import TrainDataLoader, DeviceTrainDataLoader, FullSortEvalDataLoader, NegSampleEvalDataLoader
    train, valid, test = dataset.build()
    eval_dist, n_eval_neg = parse_eval_mode((config['eval_args'] or {}).get('mode', 'full'))
    eval_dist = None if eval_dist == 'full' else eval_dist
    train_dist = parse_neg_sampling(config)
    if str(config.get('model', '')) == 'AcBERT4Rec':
        train_dist = None                        # its masked-item loss draws its own negatives (acbert4rec.py:89-93)
    samplers = build_neg_samplers(config, (train, valid, test), train_dist, eval_dist) if (train_dist or eval_dist) else (None,) * 3
    # training data resident in HBM with the epoch shuffle on the device (f-2) unless `device_resident_data: False`
    train_loader = (DeviceTrainDataLoader if device_resident_training(config) else TrainDataLoader)(
        config, train, shuffle=True, **({'neg_sampler': samplers[0]} if samplers[0] is not None else {}))
    if eval_dist is None:
        return (train_loader, FullSortEvalDataLoader(config, valid), FullSortEvalDataLoader(config, test))
    return (train_loader, NegSampleEvalDataLoader(config, valid, samplers[1], n_eval_neg),
            NegSampleEvalDataLoader(config, test, samplers[2], n_eval_neg))
