"""Top-k metrics on the [n_users, k+1] int matrix the collector builds (hit flags + pos_len):
mirrors recbole/evaluator/metrics.py:39-202, base_metric.py:43-80, evaluator.py:16-42.
Host side, numpy fp64, vectorised (the reference loops over users in MRR/NDCG).

GAUC and the item-distribution metrics (RecBole 1.0.1 metrics.py GAUC, ItemCoverage, AveragePopularity, GiniIndex,
ShannonEntropy, TailPercentage) are finalised here from what the evaluation kernels hand over instead of the [B, V] score matrix:
GAUC from per-user rank counts (G = items scoring above the positive, E = items tied with it, user_len = finite scores), the others
from the top-k item ids and the training item counts.  bincount / unique replace the reference's per-user loops."""
from collections import OrderedDict

import numpy as np


def _hit(pos, pos_len):
    return (np.cumsum(pos, axis=1) > 0).astype(int)


def _mrr(pos, pos_len):
    idx = pos.argmax(axis=1)
    has = pos[np.arange(pos.shape[0]), idx] > 0
    rr = np.where(has, 1.0 / (idx + 1), 0.0)
    k = pos.shape[1]
    return np.where(np.arange(k)[None, :] >= idx[:, None], rr[:, None], 0.0)


def _recall(pos, pos_len):
    return np.cumsum(pos, axis=1) / pos_len.reshape(-1, 1)


def _precision(pos, pos_len):
    return pos.cumsum(axis=1) / np.arange(1, pos.shape[1] + 1)


def _ndcg(pos, pos_len):
    k = pos.shape[1]
    ranks = np.arange(1, k + 1, dtype=np.float64)
    disc = 1.0 / np.log2(ranks + 1)
    idcg_full = np.cumsum(disc)
    idcg_len = np.minimum(pos_len, k).astype(np.int64)
    col = np.minimum(np.arange(k)[None, :], idcg_len[:, None] - 1)      # idcg[row, idx:] = idcg[row, idx-1]
    idcg = idcg_full[col]
    dcg = np.cumsum(np.where(pos, disc[None, :], 0.0), axis=1)
    return dcg / idcg


def _map(pos, pos_len):
    k = pos.shape[1]
    pre = pos.cumsum(axis=1) / np.arange(1, k + 1)
    sum_pre = np.cumsum(pre * pos.astype(np.float64), axis=1)
    actual = np.minimum(pos_len, k).astype(np.int64)
    ranges = np.minimum(np.arange(1, k + 1)[None, :], actual[:, None])
    return sum_pre / ranges


METRICS = {'hit': _hit, 'mrr': _mrr, 'recall': _recall, 'ndcg': _ndcg, 'precision': _precision, 'map': _map}
ITEM_METRICS = ('itemcoverage', 'averagepopularity', 'giniindex', 'shannonentropy', 'tailpercentage')
POPULARITY_METRICS = ('averagepopularity', 'tailpercentage')        # need the training item counts (data.count_items)
RANK_METRICS = ('gauc',)
VALUE_METRICS = ('auc', 'logloss', 'mae', 'rmse')


def gauc_from_counts(gt, eq, user_len):
    """metrics.py GAUC.metric_info on the collector's rec.meanrank, one positive per user.  The 1-based average rank of the positive
    in descending order is G + (E + 2) / 2 (collector.py _average_rank).  The collector's meanrank tensor is float32 (0.5 * an int
    tensor), so the arithmetic below runs in float32 exactly as the reference's does."""
    rank = np.asarray(gt, dtype=np.int64) + (np.asarray(eq, dtype=np.int64) + 2) / 2.0
    mean_rank = np.stack((rank, np.asarray(user_len, dtype=np.float64), np.ones(len(rank))), axis=1).astype(np.float32)
    pos_rank_sum, user_len_list, pos_len_list = (a.squeeze(-1) for a in np.split(mean_rank, 3, axis=1))
    neg_len_list = user_len_list - pos_len_list
    keep = (pos_len_list != 0) & (neg_len_list != 0)          # users without a negative are dropped, as the reference drops them
    user_len_list, neg_len_list, pos_len_list, pos_rank_sum = (x[keep] for x in (user_len_list, neg_len_list, pos_len_list, pos_rank_sum))
    pair_num = (user_len_list + 1) * pos_len_list - pos_len_list * (pos_len_list + 1) / 2 - pos_rank_sum
    user_auc = pair_num / (neg_len_list * pos_len_list)
    return (user_auc * pos_len_list).sum() / pos_len_list.sum()


def _distinct_counts(items):
    """occurrence counts of the distinct ids of an id matrix, ascending (Counter(...).values() sorted)"""
    _, c = np.unique(items, return_counts=True)
    return np.sort(c)


def _item_metric(m, items, k, n_items, item_counts, tail_mask):
    """value of item-distribution metric m at cut-off k from the [n_users, kmax] top-k id matrix"""
    rk = items[:, :k]
    if m == 'itemcoverage':
        return np.unique(rk).shape[0] / n_items
    if m == 'giniindex':
        c = _distinct_counts(rk)
        idx = np.arange(n_items - c.shape[0] + 1, n_items + 1)
        return np.sum((2 * idx - n_items - 1) * c) / (rk.shape[0] * rk.shape[1]) / n_items
    if m == 'shannonentropy':
        p = _distinct_counts(rk) / (rk.shape[0] * rk.shape[1])
        return float(np.sum(-p * np.log(p))) / p.shape[0]
    table = item_counts if m == 'averagepopularity' else tail_mask
    ids = items.astype(np.int64)
    inside = (ids >= 0) & (ids < table.shape[0])
    value = np.where(inside, table[np.clip(ids, 0, table.shape[0] - 1)], 0)
    avg = (value.cumsum(axis=1) / np.arange(1, value.shape[1] + 1)).mean(axis=0)
    return float(avg[k - 1])


def tail_items(item_counts, tail_ratio):
    """metrics.py TailPercentage.get_tail: the counter's items (count > 0) with count <= tail_ratio when tail_ratio > 1, else the
    first max(int(n * tail_ratio), 1) of them sorted by (count, id).  -> boolean mask over item ids"""
    cnt = np.asarray(item_counts, dtype=np.int64)
    ids = np.nonzero(cnt > 0)[0]
    mask = np.zeros(cnt.shape[0], dtype=bool)
    if tail_ratio > 1:
        mask[ids[cnt[ids] <= tail_ratio]] = True
    elif ids.shape[0]:
        order = np.lexsort((ids, cnt[ids]))
        mask[ids[order[:max(int(ids.shape[0] * tail_ratio), 1)]]] = True
    return mask


class Evaluator(object):
    """evaluator.py:16-42: evaluate(rec_topk) -> OrderedDict('metric@k' -> rounded mean over users).  GAUC needs rank counts,
    the item-distribution metrics the top-k ids (and the two popularity metrics the training item counts): see evaluate()."""

    def __init__(self, config):
        self.metrics = [m.lower() for m in config['metrics']]
        for m in self.metrics:
            if m in VALUE_METRICS:
                raise NotImplementedError('metric [%s] is a value metric: it needs labelled evaluation, which this trainer does not run '
                                          '(full-sort and sampled-candidate ranking only)' % m)
            if m not in METRICS and m not in ITEM_METRICS and m not in RANK_METRICS:
                raise NotImplementedError('metric [%s] is outside the AC-SASRec evaluation path (top-k ranking, GAUC and '
                                          'item-distribution metrics)' % m)
        self.topk = list(config['topk'])
        self.decimal_place = config['metric_decimal_place'] if config['metric_decimal_place'] is not None else 4
        try:
            tail = config['tail_ratio']
        except (KeyError, TypeError):
            tail = None
        self.tail_ratio = 0.1 if tail is None or tail <= 0 else tail          # metrics.py TailPercentage.__init__
        self.need_counts = any(m in RANK_METRICS for m in self.metrics)
        self.need_items = any(m in ITEM_METRICS for m in self.metrics)
        self.need_item_counts = any(m in POPULARITY_METRICS for m in self.metrics)

    def evaluate(self, rec_topk, counts=None, user_len=None, items=None, n_items=None, item_counts=None):
        """rec_topk [n_users, kmax+1] hit flags + pos_len; for GAUC counts [n_users, 2] (G, E) and user_len [n_users] (or one
        number); for the item-distribution metrics items [n_users, kmax] (rec.items), n_items (data.num_items, padding id 0
        included) and, for AveragePopularity / TailPercentage, item_counts [>= n_items] (the training rows per target item)."""
        rec = np.asarray(rec_topk)
        pos = rec[:, :-1].astype(bool)
        pos_len = rec[:, -1].astype(np.int64)
        if self.need_counts and counts is None:
            raise ValueError('GAUC needs the rank counts of the positive items')
        if self.need_items and (items is None or n_items is None):
            raise ValueError('the item-distribution metrics need the top-k item ids and the number of items')
        if self.need_item_counts and item_counts is None:
            raise ValueError('AveragePopularity / TailPercentage need the training item counts')
        if items is not None:
            items = np.asarray(items)
        tail_mask = tail_items(item_counts, self.tail_ratio) if 'tailpercentage' in self.metrics else None
        cnt_table = np.asarray(item_counts, dtype=np.int64) if item_counts is not None else None
        out = OrderedDict()
        for m in self.metrics:
            if m in RANK_METRICS:
                c = np.asarray(counts)
                ul = np.broadcast_to(np.asarray(user_len), (c.shape[0],))
                out[m] = round(float(gauc_from_counts(c[:, 0], c[:, 1], ul)), self.decimal_place)
                continue
            if m in ITEM_METRICS:
                for k in self.topk:
                    out['%s@%d' % (m, k)] = round(float(_item_metric(m, items, k, n_items, cnt_table, tail_mask)), self.decimal_place)
                continue
            avg = METRICS[m](pos, pos_len).mean(axis=0)
            for k in self.topk:
                out['%s@%d' % (m, k)] = round(float(avg[k - 1]), self.decimal_place)
        return out
